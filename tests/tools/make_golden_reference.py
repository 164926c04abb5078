"""Generate tests/golden/reference_modules.pt and tests/golden/reference_datasets.npz from the UNMODIFIED reference
(a checkout of andrewjong/SwapNet named by SWAPNET_REFERENCE, see oracle/ref_harness.py).

    SWAPNET_REFERENCE=/path/to/SwapNet python tests/tools/make_golden_reference.py

reference_modules.pt: the reference's WarpModule, define_D("basic") and TextureModule (pix2pix) forward in eval mode
and its PerceptualLoss(use_style=True) with the seeded-random VGG16 stand-in, all converted to float64 so that the
stored numbers do not depend on which CPU kernels a host picks (float32 results move by ~1e-5 between oneDNN's
kernels).  Each output is kept as a strided subsample plus float64 checksums of the whole tensor; the state_dict keys
and init checksums of the seed-3 WarpModule pin the parameter containers.
reference_datasets.npz: the reference's `get_transforms` (its repr) and `per_channel_transform` on a 96x96 label map for
three seeds (output + RNG digest afterwards), and `decompress_cloth_segment` of a stored 48x40 label map.
reference_warp_dataset.json: per --load_size/--crop_size, mode and sample, the RNG digest and the sha256 of the input
and target cloth tensors the reference's WarpDataset yields on tests/test_dropin_launcher.py's synthetic dataset
(its probe asserts that the warp_b200 plugin's tensors equal them before they are stored).
reference_texture_dataset.json: the same for the reference's TextureDataset per --load_size, file and seed: sha256 of
input_textures, target_textures, rois and the one-hot cloths.
Consumed by tests/test_oracle_cpu.py, tests/test_augment_cpu.py and tests/test_dropin_launcher.py.
"""
import json
import os
import random
import sys
import tempfile
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torchvision

from oracle import augment as A
from oracle import ref_harness as RH

RH.import_reference()
import modules.losses.perceptual as P  # noqa: E402  (the reference's)
from datasets import get_transforms  # noqa: E402
from datasets.data_utils import decompress_cloth_segment, per_channel_transform  # noqa: E402
from modules import init_weights  # noqa: E402
from modules.discriminators import define_D  # noqa: E402
from modules.swapnet_modules import TextureModule, WarpModule  # noqa: E402

from test_augment_cpu import label_map, rng_digest  # noqa: E402
from test_engine_gpu import synth_texture_batch, synth_warp_batch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def checksums(t):
    return (float(t.double().sum()), float(t.double().abs().sum()))


def sd_checksums(sd):
    return {k: checksums(v) for k, v in sd.items()}


def kept(t, step):
    """What the tests compare: every `step`-th pixel of the tensor plus checksums of all of it."""
    return dict(sub=t[..., ::step, ::step].clone(), sums=checksums(t), shape=tuple(t.shape))


def modules_fixture():
    gold = {}
    torch.manual_seed(0)
    G = WarpModule(); init_weights(G, "kaiming")
    D = define_D(22, 64, "basic", 3, "instance"); init_weights(D, "kaiming")
    G.double().eval(); D.double().eval()
    body, inp, _ = synth_warp_batch(2, 64)
    with torch.no_grad():
        fakes = G(body.double(), inp.double())
        pred = D(torch.cat((body.double(), fakes), 1))
    gold["warp_init"] = sd_checksums(G.state_dict())
    gold["disc_init"] = sd_checksums(D.state_dict())
    gold["warp"], gold["disc"] = kept(fakes, 4), kept(pred, 1)
    torch.manual_seed(0)
    T = TextureModule(3, 19, 12, "instance", 0.5, "pix2pix", 128); init_weights(T, "kaiming")
    gold["texture_init"] = sd_checksums(T.state_dict())
    T.double().eval()
    tex, rois, cloth, _ = synth_texture_batch(2, 128)
    with torch.no_grad():
        gold["texture"] = kept(T(tex.double(), rois.double(), cloth.double()), 8)
    torch.manual_seed(3)
    a = WarpModule(); init_weights(a, "kaiming")
    gold["seed3_keys"] = list(a.state_dict())
    gold["seed3_init"] = sd_checksums(a.state_dict())

    def seeded(pretrained=False, **kw):
        with torch.random.fork_rng():
            torch.manual_seed(1234)
            return torchvision.models.vgg16(weights=None)

    orig = P.vgg16
    P.vgg16 = seeded          # perceptual.py:26 calls vgg16(pretrained=True): a download
    try:
        crit = P.PerceptualLoss(use_style=True).double()
    finally:
        P.vgg16 = orig
    g = torch.Generator().manual_seed(5)
    out = torch.rand(2, 3, 64, 64, generator=g).double().requires_grad_()
    tgt = torch.rand(2, 3, 64, 64, generator=g).double()
    c, s = crit(out, tgt)
    (c * 20 + s * 1e-8).backward()
    gold["perceptual"] = dict(content=float(c), style=float(s), grad=kept(out.grad, 4))
    return gold


def datasets_fixture():
    out = {}
    names = ("hflip", "vflip", "affine", "perspective")
    tf = get_transforms(Namespace(input_transforms=names))
    out["transforms"] = np.array(",".join(names))
    out["transforms_repr"] = np.array(repr(tf))
    cloth = torch.from_numpy(A.onehot(label_map(96, 96, 7), 19))
    for seed in (0, 1, 2):
        random.seed(seed); torch.manual_seed(seed)
        out[f"seed{seed}_out"] = per_channel_transform(cloth, tf).numpy()
        out[f"seed{seed}_rng"] = np.array(rng_digest())
    from scipy import sparse

    with tempfile.TemporaryDirectory() as d:
        fname = os.path.join(d, "cloth.npz")
        sparse.save_npz(fname, sparse.csc_matrix(label_map(48, 40, 9).astype(np.int64)))
        out["decompressed_48x40"] = decompress_cloth_segment(fname, 19).numpy()
    return out


def warp_dataset_fixture():
    import pathlib

    from test_dropin_launcher import WARP_CONFIGS, run_warp_probe

    with tempfile.TemporaryDirectory() as d:
        got = run_warp_probe(pathlib.Path(d), RH.REF)
    assert all(g["same"] == [True] * 6 for g in got)
    return {f"{load}/{crop}": g["digests"] for (load, crop, _), g in zip(WARP_CONFIGS, got)}


def texture_dataset_fixture():
    import pathlib

    from test_dropin_launcher import TEXTURE_LOAD_SIZES, run_texture_probe

    with tempfile.TemporaryDirectory() as d:
        got = run_texture_probe(pathlib.Path(d), RH.REF)
    assert all(g["same"] == [True] * 4 for g in got)
    return {size: g["digests"] for size, g in zip(TEXTURE_LOAD_SIZES, got)}


if __name__ == "__main__":
    path = os.path.join(OUT, "reference_modules.pt")
    torch.save(modules_fixture(), path)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(OUT, "reference_datasets.npz")
    np.savez_compressed(path, **datasets_fixture())
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(OUT, "reference_warp_dataset.json")
    with open(path, "w") as f:
        json.dump(warp_dataset_fixture(), f, indent=1)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(OUT, "reference_texture_dataset.json")
    with open(path, "w") as f:
        json.dump(texture_dataset_fixture(), f, indent=1)
    print("wrote", path, os.path.getsize(path), "bytes")

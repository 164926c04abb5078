"""CPU tests of the device-side input pipeline's host half and of its oracle (SURVEY §8 f4).

  * oracle/augment.py (numpy restatement of Pillow's resampling) is pinned bit-exactly against Pillow / torchvision
    themselves and against what the reference's own `per_channel_transform(get_transforms(opt))` produced
    (tests/golden/augment_64.npz, tests/golden/reference_datasets.npz);
  * swapnet_b200.data.draw_channel_ops makes the reference's random draws without touching pixels: same ops, and the
    python `random` / torch generators end in the same state.
The device kernel is compared with the same oracle in tests/test_augment_gpu.py.
"""
import hashlib
import os
import random
from argparse import Namespace

import numpy as np
import pytest
import torch
from PIL import Image
from torchvision import transforms as T
from torchvision.transforms import functional as TF

from oracle import augment as A
from swapnet_b200 import data as D

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "augment_64.npz")
REFERENCE_DATASETS = os.path.join(os.path.dirname(__file__), "golden", "reference_datasets.npz")
SIZES = [(64, 64), (128, 96), (37, 53), (512, 512)]


def reference_transform(names):
    """datasets/__init__.py:88-110 `get_transforms` restated with the same torchvision objects;
    `test_matches_the_reference_function` checks it against the real one."""
    tl = []
    every = "all" in names
    if every or "vflip" in names:
        tl.append(T.RandomVerticalFlip())
    if every or "hflip" in names:
        tl.append(T.RandomHorizontalFlip())
    if every or "affine" in names:
        tl.append(T.RandomAffine(degrees=10, translate=(0.1, 0.1), scale=(0.8, 1.2), shear=20))
    if every or "perspective" in names:
        tl.append(T.RandomPerspective())
    return T.RandomOrder(tl)


def pil_per_channel(planes: np.ndarray, tf) -> np.ndarray:
    """datasets/data_utils.py:346-361 through Pillow / torchvision themselves."""
    out = np.zeros_like(planes)
    for i in range(planes.shape[0]):
        out[i] = np.array(tf(Image.fromarray(planes[i])))
    return out


def label_map(h, w, seed):
    g = np.random.default_rng(seed)
    return g.integers(0, 19, ((h + 7) // 8, (w + 7) // 8)).repeat(8, 0).repeat(8, 1)[:h, :w].astype(np.uint8)


def rng_digest() -> str:
    h = hashlib.sha256()
    h.update(np.asarray(random.getstate()[1], dtype=np.uint64).tobytes())
    h.update(torch.get_rng_state().numpy().tobytes())
    return h.hexdigest()


def plane(h, w, seed, binary):
    g = np.random.default_rng(seed)
    if binary:
        return (label_map(h, w, seed) == 3).astype(np.float32)
    return g.random((h, w)).astype(np.float32)


@pytest.mark.parametrize("binary", [True, False])
def test_oracle_affine_nearest_is_pillow(binary):
    g = np.random.default_rng(5)
    for trial in range(40):
        h, w = SIZES[trial % len(SIZES)]
        img = plane(h, w, trial, binary)
        m = TF._get_inverse_affine_matrix([w * 0.5, h * 0.5], g.uniform(-10, 10),
                                          [int(round(g.uniform(-.1 * w, .1 * w))), int(round(g.uniform(-.1 * h, .1 * h)))],
                                          g.uniform(.8, 1.2), [g.uniform(-20, 20), 0.0])
        ref = np.array(Image.fromarray(img).transform((w, h), Image.AFFINE, m, Image.NEAREST, fillcolor=0))
        assert np.array_equal(A.affine_nearest(img, m), ref), trial


@pytest.mark.parametrize("binary", [True, False])
def test_oracle_perspective_bilinear_is_pillow(binary):
    for trial in range(40):
        h, w = SIZES[trial % len(SIZES)]
        img = plane(h, w, trial, binary)
        torch.manual_seed(trial)
        c = TF._get_perspective_coeffs(*T.RandomPerspective.get_params(w, h, 0.5))
        ref = np.array(Image.fromarray(img).transform((w, h), Image.PERSPECTIVE, c, Image.BILINEAR, fillcolor=0))
        assert np.array_equal(A.perspective_bilinear(img, c), ref), trial


def test_oracle_flips_are_pillow():
    img = plane(37, 53, 1, False)
    assert np.array_equal(A.hflip(img), np.array(TF.hflip(Image.fromarray(img))))
    assert np.array_equal(A.vflip(img), np.array(TF.vflip(Image.fromarray(img))))


@pytest.mark.parametrize("names", [("hflip", "vflip", "affine", "perspective"), ("affine",), ("perspective", "hflip")])
@pytest.mark.parametrize("size", [(64, 64), (40, 56)])
def test_host_draws_plus_oracle_equal_the_pillow_pipeline(names, size):
    h, w = size
    tf = reference_transform(names)
    planes = A.onehot(label_map(h, w, 3), 19)
    for seed in range(4):
        random.seed(seed); torch.manual_seed(seed)
        ref = pil_per_channel(planes, tf)
        state = rng_digest()
        random.seed(seed); torch.manual_seed(seed)
        ops = D.draw_channel_ops(tf, 19, w, h)
        assert rng_digest() == state, "the host draws must advance python random and torch exactly like the reference"
        assert np.array_equal(A.per_channel_transform(planes, ops), ref)


def test_matches_the_reference_function():
    """The reference's own `get_transforms` + `per_channel_transform` on a 96x96 label map, stored by
    tests/tools/make_golden_reference.py: `reference_transform` builds the same transform object, and the host draws +
    oracle give the same pixels and leave both generators in the same state."""
    z = np.load(REFERENCE_DATASETS)
    tf = reference_transform(tuple(str(z["transforms"]).split(",")))
    assert repr(tf) == str(z["transforms_repr"])
    cloth = A.onehot(label_map(96, 96, 7), 19)
    for seed in (0, 1, 2):
        random.seed(seed); torch.manual_seed(seed)
        ops = D.draw_channel_ops(tf, 19, 96, 96)
        assert rng_digest() == str(z[f"seed{seed}_rng"])
        assert np.array_equal(A.per_channel_transform(cloth, ops), z[f"seed{seed}_out"])


def test_golden_fixture_from_the_reference():
    z = np.load(GOLDEN)
    for name in ("all_64", "all_40x56", "affine_64", "flips_64"):
        lab, ref, seed = z[name + "_labels"], z[name + "_out"], int(z[name + "_seed"])
        tf = reference_transform(tuple(str(z[name + "_transforms"]).split(",")))
        random.seed(seed); torch.manual_seed(seed)
        ops = D.draw_channel_ops(tf, 19, lab.shape[1], lab.shape[0])
        assert rng_digest() == str(z[name + "_rng"]), name
        assert np.array_equal(A.per_channel_transform(A.onehot(lab, 19), ops), ref), name


def test_op_table_layout_and_refusals():
    ops = [[(D.AUG_HFLIP, ())], [], [(D.AUG_AFFINE_NEAREST, (1, 2, 3, 4, 5, 6)), (D.AUG_VFLIP, ())]]
    table, max_ops = D.encode_ops(ops)
    assert max_ops == 2 and table.shape == (3, 2) and table.dtype.itemsize == 72
    assert table.dtype.fields["kind"][1] == 0 and table.dtype.fields["nops"][1] == 4 and table.dtype.fields["p"][1] == 8
    assert table["nops"].tolist() == [[1, 1], [0, 0], [2, 2]] and table["kind"][2].tolist() == [3, 2]
    assert table["p"][2, 0, :6].tolist() == [1, 2, 3, 4, 5, 6]
    assert D.encode_ops([[]])[0].shape == (1, 1)
    with pytest.raises(NotImplementedError):           # Pillow's pure-scale path is not restated
        D._affine_op([1.1, 0.0, 3.0, 0.0, 0.9, -2.0], 64, 64)
    with pytest.raises(NotImplementedError):
        D.draw_channel_ops(T.ColorJitter(), 1, 8, 8)
    with pytest.raises(NotImplementedError):
        D.draw_channel_ops(T.RandomAffine(10, interpolation=T.InterpolationMode.BILINEAR), 1, 8, 8)
    assert D.draw_channel_ops(None, 3, 8, 8) == [[], [], []]
    t = D.OpTable([ops[:2], ops[1:]], pin=False)
    assert (t.batch, t.channels, t.stride, t.max_ops, t.nbytes) == (2, 2, 2, 2, 2 * 2 * 2 * 72)
    with pytest.raises(RuntimeError):                  # no CPU path
        D.ClothAugmenter(None, 2).apply(torch.zeros(1, 8, 8, dtype=torch.uint8), [[[], []]])


def test_load_label_map_equals_the_reference_decompression(tmp_path):
    from scipy import sparse

    lab = label_map(48, 40, 9)
    fname = str(tmp_path / "cloth.npz")
    sparse.save_npz(fname, sparse.csc_matrix(lab.astype(np.int64)))      # data_utils.py:311-327 compress_and_save_cloth
    got = D.load_label_map(fname)
    assert got.dtype == np.uint8 and np.array_equal(got, lab)
    # the reference's decompress_cloth_segment(fname, 19) of the same file (tests/tools/make_golden_reference.py)
    assert np.array_equal(A.onehot(got, 19), np.load(REFERENCE_DATASETS)["decompressed_48x40"])


def test_kernel_source_run_on_the_host_equals_oracle(tmp_path):
    """csrc/augment.cu's device code compiled for the host (tests/tools/kernel_host_shim.py): same pixels as the
    oracle for label-map and dense sources, 0-4 ops per plane (the GPU run of the real kernel: test_augment_gpu.py)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "tools"))
    import kernel_host_shim

    lib = kernel_host_shim.build(str(tmp_path))
    if lib is None:
        pytest.skip("no g++")

    def run(labels, dense, sample_ops, c):
        table, max_ops = D.encode_ops([o for s in sample_ops for o in s])
        table = np.ascontiguousarray(table)
        src = labels if labels is not None else dense
        n, (h, w) = src.shape[0], src.shape[-2:]
        out, tmp = np.full((n, c, h, w), -7, np.float32), np.full((n, c, h, w), -9, np.float32)
        lib.run(labels.ctypes.data if labels is not None else None, dense.ctypes.data if dense is not None else None,
                n, c, h, w, table.ctypes.data, table.shape[1], max_ops, out.ctypes.data, tmp.ctypes.data)
        return out

    tf = reference_transform(("hflip", "vflip", "affine", "perspective"))
    for h, w in ((64, 64), (33, 130)):
        labs = np.stack([label_map(h, w, 20 + b) for b in range(2)])
        random.seed(1); torch.manual_seed(1)
        sample_ops = [D.draw_channel_ops(tf, 19, w, h) for _ in range(2)]
        assert {len(o) for s in sample_ops for o in s} >= {1, 2, 3}
        got = run(labs, None, sample_ops, 19)
        for b in range(2):
            assert np.array_equal(got[b], A.per_channel_transform(A.onehot(labs[b], 19), sample_ops[b]))
    dense = np.random.default_rng(3).random((1, 19, 40, 56)).astype(np.float32)
    random.seed(2); torch.manual_seed(2)
    sample_ops = [D.draw_channel_ops(tf, 19, 56, 40)]
    sample_ops[0][0] = []                                   # a plane without ops: straight copy
    assert np.array_equal(run(None, dense, sample_ops, 19)[0], A.per_channel_transform(dense[0], sample_ops[0]))


def test_sample_format_round_trip_and_guards():
    """`encode_sample` (what `--dataset warp_b200` puts into a sample) -> default collate -> `OpTable.from_collated`."""
    tf = reference_transform(("hflip", "vflip", "affine", "perspective"))
    random.seed(3); torch.manual_seed(3)
    per_sample = [D.draw_channel_ops(tf, 19, 64, 64) for _ in range(3)]
    stacked = torch.utils.data.default_collate([{"input_ops": D.encode_sample(o, 4)} for o in per_sample])["input_ops"]
    t = D.OpTable.from_collated(stacked, 19)
    want = D.OpTable(per_sample, pin=False)
    assert (t.batch, t.channels, t.stride) == (3, 19, 4) and t.max_ops == want.max_ops
    a = t.host.numpy().view(D.OP_DTYPE).reshape(57, 4)
    b = want.host.numpy().view(D.OP_DTYPE).reshape(57, want.stride)
    for f in ("kind", "nops", "p"):
        assert np.array_equal(a[f][:, :want.stride], b[f]), f
    assert not a["kind"][:, want.stride:].any()
    with pytest.raises(NotImplementedError):                     # more ops than the sample format has slots for
        D.encode_sample([[(D.AUG_HFLIP, ())] * 5], 4)
    bad = stacked.clone()
    bad.numpy().view(D.OP_DTYPE)["nops"][0] = 9
    with pytest.raises(ValueError):
        D.OpTable.from_collated(bad, 19)


def test_datasets_overlay_refuses_to_load_without_the_reference_package(tmp_path):
    """dropin/datasets is an overlay of the reference's package: imported on its own it must say so, not half-work."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); import datasets" % os.path.join(root, "dropin")],
                       cwd=str(tmp_path), capture_output=True, text=True, env={**os.environ, "PYTHONPATH": ""})
    assert r.returncode != 0 and "overlays the reference's `datasets` package" in r.stderr

"""The drop-in boundary, end to end on the CPU: a checkout's unmodified `train.py` started through
`python -m swapnet_b200.run` resolves `models` to this repo's plugins, parses its options through them
(options/base_options.py:171-186), builds the checkout's dataset from files on disk and reaches the plugin's
constructor — which, on a box without a GPU, refuses to run (there is no CPU fallback).  On a GPU box the same command
trains (tests/test_engine_gpu.py::test_train_loop_protocol restates train.py:31-116 there).  The checkout is the
reference's when SWAPNET_REFERENCE names one, else tests/tools/standin_swapnet (the same train.py / options / datasets
surface, written for these tests).  Either way the dataset plugins must yield what the reference's own WarpDataset and
TextureDataset yield on the same files and seeds (tests/golden/reference_{warp,texture}_dataset.json)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STANDIN = os.path.join(ROOT, "tests", "tools", "standin_swapnet")
REF = os.path.abspath(os.environ["SWAPNET_REFERENCE"]) if os.environ.get("SWAPNET_REFERENCE") else STANDIN
STUBS = os.path.join(ROOT, "tests", "tools", "ref_stubs")
WARP_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_warp_dataset.json")
TEXTURE_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_texture_dataset.json")


def make_dataset(root, n=2, size=64):
    """A tiny dataset in the reference's on-disk format: cloth/*.npz (scipy CSC label maps, data_utils.py:311-327),
    body/*.jpg, texture/*.jpg, normalization_stats.json (json lines indexed by `path`, data_utils.py:30-38)."""
    from PIL import Image
    from scipy import sparse

    rng = np.random.RandomState(0)
    for d in ("cloth", "body", "texture"):
        os.makedirs(os.path.join(root, d), exist_ok=True)
    for i in range(n):
        lab = np.kron(rng.randint(0, 19, (size // 16, size // 16)), np.ones((16, 16), dtype=np.int64))
        sparse.save_npz(os.path.join(root, "cloth", f"s{i}.npz"), sparse.csc_matrix(lab))
        for d in ("body", "texture"):
            Image.fromarray(rng.randint(0, 255, (size, size, 3), dtype=np.uint8)).save(os.path.join(root, d, f"s{i}.jpg"))
    with open(os.path.join(root, "rois.csv"), "w") as f:          # 12 ROI rows per file id (texture_dataset.py:73-76,117-119)
        f.write("id,xmin,ymin,xmax,ymax\n")
        for i in range(n):
            for k in range(12):
                x0, y0 = rng.randint(0, size // 2, 2)
                f.write(f"s{i},{x0},{y0},{x0 + rng.randint(1, size // 2)},{y0 + rng.randint(1, size // 2)}\n")
    with open(os.path.join(root, "normalization_stats.json"), "w") as f:
        for k in ("body", "texture", "cloth"):
            f.write(json.dumps({"path": k, "means": [0.5, 0.5, 0.5], "stds": [0.25, 0.25, 0.25]}) + "\n")


def run(cmd, cwd, extra_path=()):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([*extra_path, ROOT, STUBS, os.path.join(ROOT, "tests")])
    env["CUDA_VISIBLE_DEVICES"] = ""
    return subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=600)


def test_plain_python_train_py_resolves_the_reference_models_package(tmp_path):
    """Why a launcher is needed: `python script.py` puts the script's directory first, so PYTHONPATH cannot shadow
    the checkout's `models` package (a stand-in checkout: a script next to a `models` package)."""
    checkout = tmp_path / "checkout"
    (checkout / "models").mkdir(parents=True)
    (checkout / "models" / "__init__.py").write_text("")
    (checkout / "train.py").write_text("import models\nprint(models.__file__)\n")
    r = run([sys.executable, str(checkout / "train.py")], cwd=str(tmp_path), extra_path=[os.path.join(ROOT, "dropin")])
    assert r.returncode == 0 and r.stdout.strip().startswith(str(checkout)), (r.stdout, r.stderr[-2000:])


@pytest.mark.parametrize("dataset", [None, "warp_b200"])
def test_launcher_runs_unmodified_train_py_through_the_plugin(tmp_path, dataset):
    """dataset=None: the reference's own WarpDataset (through the dropin/datasets overlay, which must be transparent);
    "warp_b200": the plugin dataset found by the reference's registry (device-side augmentation, f4)."""
    data = tmp_path / "data"
    make_dataset(str(data))
    ck = tmp_path / "ck"
    r = run([sys.executable, "-m", "swapnet_b200.run", "train.py", "--name", "t", "--model", "warp", "--dataroot",
             str(data), "--checkpoints_dir", str(ck), "--display_id", "0", "--batch_size", "1", "--load_size", "64",
             "--crop_size", "64", "--num_workers", "0", "--no_confirm", "--gpu_id", "0", "--n_epochs", "1",
             *(["--dataset", dataset] if dataset else [])], cwd=REF)
    out = r.stdout + r.stderr
    assert ("dataset [WarpB200Dataset] was created" if dataset else "dataset [WarpDataset] was created") in out, out[-3000:]
    # options parsed through the plugin: our extra flag is in the printed / stored option table (train_options.py)
    assert "b200_precision" in out, out[-3000:]
    assert "The number of training images = 2" in out, out[-3000:]
    # ... and the model constructor that refused is OURS (no GPU here, no CPU fallback)
    assert r.returncode != 0
    assert "swapnet_b200 models run on a CUDA device only" in out, out[-3000:]
    assert os.path.join("swapnet_b200", "models", "base_model.py") in out


def test_launcher_option_defaults_match_the_reference_parser(tmp_path):
    """TrainOptions().parse() through the plugin yields the reference's defaults for every flag that reaches the hot
    path (SURVEY App. D), for both models."""
    probe = tmp_path / "probe.py"
    probe.write_text(
        "import sys, json\n"
        "import models\n"
        "from options.train_options import TrainOptions\n"
        "opt = TrainOptions().parse(print_options=False) if 'print_options' in TrainOptions.parse.__code__.co_varnames"
        " else TrainOptions().parse()\n"
        "keys = ['lr','d_lr','weight_decay','d_weight_decay','b1','b2','gan_mode','gan_label_mode','norm','init_type',"
        "'lambda_gan','lambda_discriminator','discriminator','optimizer_G','optimizer_D','b200_precision']\n"
        "extra = {'warp': ['warp_mode','lambda_ce'], 'texture': ['lambda_l1','lambda_content','lambda_style','netG']}\n"
        "print('PROBE', json.dumps({'file': models.__file__, **{k: getattr(opt, k) for k in keys + extra[opt.model]}}))\n")
    want = dict(lr=1e-4, d_lr=4e-4, weight_decay=0, d_weight_decay=0.01, b1=0.9, b2=0.999, gan_mode="vanilla",
                gan_label_mode="smooth", norm="instance", init_type="kaiming", lambda_gan=1.0, lambda_discriminator=1.0,
                discriminator="basic", optimizer_G="AdamW", optimizer_D="AdamW", b200_precision="fp32x3")
    extra = dict(warp=dict(warp_mode="gan", lambda_ce=100), texture=dict(lambda_l1=10, lambda_content=20,
                                                                         lambda_style=1e-8, netG="swapnet"))
    data = tmp_path / "data"
    make_dataset(str(data))
    # the probe must live in the checkout directory for Python's script start-up rule to bite: emulate by cwd + path
    for model in ("warp", "texture"):
        r = run([sys.executable, "-m", "swapnet_b200.run", str(probe), "--name", "p", "--model", model, "--dataroot",
                 str(data), "--checkpoints_dir", str(tmp_path / "ck"), "--no_confirm"], cwd=REF, extra_path=[REF])
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE ")]
        assert r.returncode == 0 and line, (r.stdout[-2000:], r.stderr[-3000:])
        got = json.loads(line[-1][6:])
        assert got.pop("file").startswith(os.path.join(ROOT, "dropin")), got
        for k, v in {**want, **extra[model]}.items():
            assert got[k] == v, (model, k, got[k], v)


# stored size 64: as is; resized x2 and centre-cropped back to 64 (the reference resizes / crops AFTER the augmentation:
# a gather per axis here); resized x2 without a crop
WARP_CONFIGS = (("64", "64", 64), ("128", "64", 64), ("128", "128", 128))


def run_warp_probe(tmp_path, ref):
    """--dataset warp_b200 through the launcher from checkout `ref`, per WARP_CONFIGS: the probe's result dicts."""
    probe = tmp_path / "probe.py"
    probe.write_text(
        "import sys, json, random, hashlib\n"
        "import numpy as np, torch\n"
        "import datasets, datasets.warp_dataset, datasets.data_utils\n"
        "from options.train_options import TrainOptions\n"
        "from oracle import augment as A\n"
        "from swapnet_b200 import data as D\n"
        "opt = TrainOptions().parse()\n"
        "loader = datasets.create_dataset(opt)\n"
        "mine = loader.dataset\n"
        "ref = datasets.warp_dataset.WarpDataset(opt)\n"
        "def digest():\n"
        "    h = hashlib.sha256(); h.update(np.asarray(random.getstate()[1], dtype=np.uint64).tobytes())\n"
        "    h.update(torch.get_rng_state().numpy().tobytes()); return h.hexdigest()\n"
        "def decode(t, c):\n"
        "    tab = t.numpy().view(D.OP_DTYPE).reshape(c, -1)\n"
        "    return [[(int(tab['kind'][i, j]), tab['p'][i, j]) for j in range(int(tab['nops'][i, 0]))] for i in range(c)]\n"
        "res = dict(datasets_file=datasets.__file__, warp_dataset_file=datasets.warp_dataset.__file__,\n"
        "           data_utils_file=datasets.data_utils.__file__, cls=type(mine).__name__, n=len(mine), same=[], nops=[], digests=[])\n"
        "for mode in ('image', 'video'):\n"
        "    opt.dataset_mode = mode\n"
        "    for idx in range(len(mine)):\n"
        "        random.seed(idx); torch.manual_seed(idx); r = ref[idx]; d_ref = digest()\n"
        "        random.seed(idx); torch.manual_seed(idx); m = mine[idx]; d_mine = digest()\n"
        "        ops = decode(m['input_ops'], 19)\n"
        "        inp = torch.from_numpy(A.per_channel_transform(A.onehot(m['input_labels'].numpy(), 19), ops))\n"
        "        tgt = torch.from_numpy(A.onehot(m['target_labels'].numpy(), 19))\n"
        "        if 'resize_iy' in m:      # what WarpModel.set_input does on the device\n"
        "            inp = D.gather_rows_cols(inp, m['resize_iy'], m['resize_ix'])\n"
        "            tgt = D.gather_rows_cols(tgt, m['resize_iy'], m['resize_ix'])\n"
        "        res['gather'] = 'resize_iy' in m\n"
        "        res['nops'].append(max(len(o) for o in ops))\n"
        "        res['digests'].append([d_mine] + [hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest() for t in (inp, tgt)])\n"
        "        res['same'].append(bool(d_ref == d_mine and torch.equal(inp, r['input_cloths'])\n"
        "                           and torch.equal(tgt, r['target_cloths'])\n"
        "                           and torch.equal(m['bodys'], r['bodys']) and m['cloth_paths'] == r['cloth_paths']\n"
        "                           and m['body_paths'] == r['body_paths']))\n"
        "opt.dataset_mode = 'image'\n"
        "batch = next(iter(loader))\n"
        "res['batch'] = {k: (list(v.shape), str(v.dtype)) if hasattr(v, 'shape') else len(v) for k, v in batch.items()}\n"
        "t = D.OpTable.from_collated(batch['input_ops'], 19)\n"
        "res['table'] = [t.batch, t.channels, t.stride]\n"
        "print('PROBE', json.dumps(res))\n")
    data = tmp_path / "data"
    make_dataset(str(data), n=3)
    results = []
    for load, crop, _ in WARP_CONFIGS:
        r = run([sys.executable, "-m", "swapnet_b200.run", str(probe), "--name", "p", "--model", "warp", "--dataset",
                 "warp_b200", "--dataroot", str(data), "--checkpoints_dir", str(tmp_path / "ck"), "--no_confirm",
                 "--batch_size", "2", "--load_size", load, "--crop_size", crop, "--num_workers", "0",
                 "--shuffle_data", ""], cwd=ref,            # type=bool: "" is False, the files are taken in sorted order
                extra_path=[ref])
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE ")]
        assert r.returncode == 0 and line, (r.stdout[-2000:], r.stderr[-3000:])
        results.append(json.loads(line[-1][6:]))
    return results


def test_dataset_overlay_and_warp_b200_dataset_match_the_reference_dataset(tmp_path):
    """SURVEY §8 f4 through the reference's own registry: `--dataset warp_b200` (dropin/datasets, an overlay that leaves
    every reference module in place) yields, sample by sample and with the generators in the same state afterwards, label
    maps + op tables that expand to exactly the tensors the reference's WarpDataset yields (image and video mode)."""
    got = run_warp_probe(tmp_path, REF)
    with open(WARP_DIGESTS) as f:
        gold = json.load(f)
    for (load, crop, out), g in zip(WARP_CONFIGS, got):
        assert g["datasets_file"].startswith(os.path.join(ROOT, "dropin", "datasets"))
        assert g["warp_dataset_file"].startswith(REF) and g["data_utils_file"].startswith(REF)
        assert g["cls"] == "WarpB200Dataset" and g["n"] == 3
        assert g["same"] == [True] * 6, g
        # what the reference's own WarpDataset yielded for the same files and seeds (RNG state, input, target)
        assert g["digests"] == gold[f"{load}/{crop}"], (load, crop)
        assert g["gather"] == (load != "64")
        assert max(g["nops"]) >= 3                      # the default transform set really drew something
        assert g["batch"]["input_labels"] == [[2, 64, 64], "torch.uint8"] and g["batch"]["bodys"][0] == [2, 3, out, out]
        assert g["batch"]["input_ops"] == [[2, 19 * 4 * 72], "torch.uint8"] and g["table"] == [2, 19, 4]
        if load != "64":
            assert g["batch"]["resize_iy"] == [[2, out], "torch.int64"]


TEXTURE_LOAD_SIZES = ("64", "96")


def run_texture_probe(tmp_path, ref):
    """--dataset texture_b200 through the launcher from checkout `ref`, per TEXTURE_LOAD_SIZES: the probe's result
    dicts.  Each sample is drawn twice, with seeds taken from its file id (the reference does not sort the texture
    files, so an index does not name the same file everywhere); `digests[f"{id}/{seed}"]` = sha256 of the plugin's
    input_textures, target_textures, rois and one-hot cloths."""
    probe = tmp_path / "probe.py"
    probe.write_text(
        "import sys, json, random, hashlib, os\n"
        "import numpy as np, torch\n"
        "import datasets, datasets.texture_dataset\n"
        "from options.train_options import TrainOptions\n"
        "from oracle import augment as A\n"
        "opt = TrainOptions().parse()\n"
        "loader = datasets.create_dataset(opt)\n"
        "mine, ref = loader.dataset, datasets.texture_dataset.TextureDataset(opt)\n"
        "def sha(t):\n"
        "    return hashlib.sha256(np.ascontiguousarray(t).tobytes()).hexdigest()\n"
        "same, digests = [], {}\n"
        "for idx in range(len(mine)):\n"
        "    fid = os.path.splitext(os.path.basename(mine.texture_files[idx]))[0]\n"
        "    for seed in (int(fid[1:]), int(fid[1:]) + 10):\n"
        "        random.seed(seed); torch.manual_seed(seed); r = ref[idx]\n"
        "        random.seed(seed); torch.manual_seed(seed); m = mine[idx]\n"
        "        onehot = A.onehot(m['cloths'].numpy(), 19)\n"
        "        digests[f'{fid}/{seed}'] = [sha(m[k].numpy()) for k in ('input_textures', 'target_textures', 'rois')] + [sha(onehot)]\n"
        "        same.append(bool(m['cloths'].dtype == torch.uint8 and m['cloths'].dim() == 2\n"
        "                    and np.array_equal(onehot, r['cloths'].numpy())\n"
        "                    and torch.equal(m['input_textures'], r['input_textures']) and torch.equal(m['rois'], r['rois'])\n"
        "                    and torch.equal(m['target_textures'], r['target_textures'])\n"
        "                    and m['cloth_paths'] == r['cloth_paths'] and m['texture_paths'] == r['texture_paths']))\n"
        "batch = next(iter(loader))\n"
        "print('PROBE', json.dumps(dict(cls=type(mine).__name__, same=same, digests=digests,\n"
        "      cloths=[list(batch['cloths'].shape), str(batch['cloths'].dtype)],\n"
        "      restored=datasets.texture_dataset.decompress_cloth_segment.__module__)))\n")
    data = tmp_path / "data"
    make_dataset(str(data), n=2)
    results = []
    for load_size in TEXTURE_LOAD_SIZES:
        r = run([sys.executable, "-m", "swapnet_b200.run", str(probe), "--name", "p", "--model", "texture", "--dataset",
                 "texture_b200", "--dataroot", str(data), "--checkpoints_dir", str(tmp_path / "ck"), "--no_confirm",
                 "--batch_size", "2", "--load_size", load_size, "--crop_size", load_size, "--num_workers", "0"],
                cwd=ref, extra_path=[ref])
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE ")]
        assert r.returncode == 0 and line, (r.stdout[-2000:], r.stderr[-3000:])
        results.append(json.loads(line[-1][6:]))
    return results


def test_texture_b200_dataset_matches_the_reference_dataset(tmp_path):
    """`--dataset texture_b200`: same samples as the reference's TextureDataset (textures, ROIs incl. the joint random
    flips, paths), the cloth as a uint8 label map whose one-hot expansion is the reference's tensor — also when the
    stored size differs from --load_size (nearest resize of the label plane).  Pinned to what the reference's own
    TextureDataset yields on the same files and seeds (tests/golden/reference_texture_dataset.json)."""
    got = run_texture_probe(tmp_path, REF)
    with open(TEXTURE_DIGESTS) as f:
        gold = json.load(f)
    for load_size, g in zip(TEXTURE_LOAD_SIZES, got):
        assert g["cls"] == "TextureB200Dataset" and g["same"] == [True] * 4, g
        assert g["digests"] == gold[load_size], load_size
        assert g["cloths"] == [[2, int(load_size), int(load_size)], "torch.uint8"]
        assert g["restored"] == "datasets.data_utils"           # the substitution does not outlive __getitem__

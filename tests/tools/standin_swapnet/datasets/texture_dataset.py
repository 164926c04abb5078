import csv
import os
import random

import numpy as np
import torch
import torchvision.transforms.functional as tf
from PIL import Image
from torch import nn
from torchvision import transforms

from datasets import BaseDataset
from datasets.data_utils import crop_tensors, decompress_cloth_segment, find_valid_files, get_norm_stats


def mirror(rois, lo, hi, centre):
    """Reflect the coordinate pair (columns lo, hi) about `centre`; the two swap roles."""
    out = rois.clone()
    out[:, lo], out[:, hi] = 2 * centre - rois[:, hi], 2 * centre - rois[:, lo]
    return out


class TextureDataset(BaseDataset):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        parser.add_argument("--input_transforms", nargs="+", default=("hflip", "vflip") if is_train else "none")
        return parser

    def __init__(self, opt):
        super().__init__(opt)
        self.texture_dir = os.path.join(opt.dataroot, "texture")
        self.cloth_dir = os.path.join(opt.dataroot, "cloth")
        self.texture_files = find_valid_files(self.texture_dir, [".jpg", ".png"])
        self._normalize = transforms.Normalize(*get_norm_stats(opt.dataroot, "texture"))
        self.rois = {}
        with open(os.path.join(opt.dataroot, "rois.csv")) as f:
            for row in csv.DictReader(f):
                self.rois.setdefault(row["id"], []).append([float(row[k]) for k in ("xmin", "ymin", "xmax", "ymax")])

    def __len__(self):
        return len(self.texture_files)

    def __getitem__(self, index):
        size = self.opt.load_size
        texture_file = self.texture_files[index]
        img = Image.open(texture_file).convert("RGB")
        target = self._normalize(tf.to_tensor(tf.resize(img, size)))
        file_id = os.path.splitext(os.path.basename(texture_file))[0]
        cloth_file = os.path.join(self.cloth_dir, file_id + ".npz")
        # looked up on the module at call time, like the reference (the texture_b200 plugin substitutes it)
        cloth = nn.functional.interpolate(decompress_cloth_segment(cloth_file, n_labels=19).unsqueeze(0),
                                          size=size).squeeze()
        rois = torch.from_numpy(np.rint(np.array(self.rois[file_id], np.float32) * (float(size) / img.size[0])))
        # input = target randomly flipped, vertical draw first; the ROIs (already at --load_size) are mirrored about
        # the centre of the STORED image, as the reference does
        names = self.opt.input_transforms
        w, h = img.size
        if random.random() < (0.5 if "vflip" in names or "all" in names else 0):
            img, rois = tf.vflip(img), mirror(rois, 1, 3, int(h / 2))
        if random.random() < (0.5 if "hflip" in names or "all" in names else 0):
            img, rois = tf.hflip(img), mirror(rois, 0, 2, int(w / 2))
        inp = self._normalize(tf.to_tensor(tf.resize(img, size)))
        if self.crop_bounds:
            inp, cloth, target = crop_tensors(inp, cloth, target, crop_bounds=self.crop_bounds)
        return {"texture_paths": texture_file, "input_textures": inp, "rois": rois, "cloth_paths": cloth_file,
                "cloths": cloth, "target_textures": target}

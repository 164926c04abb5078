import os
import random

from PIL import Image
from torch import nn
from torchvision import transforms

from datasets import BaseDataset
from datasets.data_utils import crop_tensors, decompress_cloth_segment, find_valid_files, get_norm_stats, per_channel_transform
from test_augment_cpu import reference_transform      # the tests' restatement of the reference's transform set

# the warp stage's default training augmentation
TRANSFORMS = ("hflip", "vflip", "affine", "perspective")


class WarpDataset(BaseDataset):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        parser.add_argument("--per_channel_transform", action="store_true", default=True)
        return parser

    def __init__(self, opt, cloth_dir=None, body_dir=None):
        super().__init__(opt)
        self.cloth_dir = cloth_dir or os.path.join(opt.dataroot, "cloth")
        self.body_dir = body_dir or os.path.join(opt.dataroot, "body")
        self.cloth_files = find_valid_files(self.cloth_dir, [".npz"])
        self._normalize_body = transforms.Normalize(*get_norm_stats(opt.dataroot, "body"))
        self.cloth_transform = reference_transform(TRANSFORMS)

    def __len__(self):
        return len(self.cloth_files)

    def _load_body(self, index):
        name = os.path.splitext(os.path.basename(self.cloth_files[index]))[0]
        body_file = os.path.join(self.body_dir, name + ".jpg")
        return body_file, self._normalize_body(transforms.ToTensor()(Image.open(body_file).convert("RGB")))

    def __getitem__(self, index):
        cloth_file = self.cloth_files[index]
        target = decompress_cloth_segment(cloth_file, self.opt.cloth_channels)
        source = target.clone()
        if self.opt.dataset_mode == "video":
            # the input is another frame of the set, drawn as the plugin draws it (index 0 wraps to the last file)
            k = random.randint(0, len(self))
            cloth_file = self.cloth_files[k - 1]
            source = decompress_cloth_segment(cloth_file, self.opt.cloth_channels)
        if self.cloth_transform:
            source = per_channel_transform(source, self.cloth_transform)
        body_file, body = self._load_body(index)
        size = self.opt.load_size
        source = nn.functional.interpolate(source.unsqueeze(0), size=size).squeeze()
        target = nn.functional.interpolate(target.unsqueeze(0), size=size).squeeze()
        body = nn.functional.interpolate(body.unsqueeze(0), size=size, mode="bilinear").squeeze()
        if self.crop_bounds:
            source, body, target = crop_tensors(source, body, target, crop_bounds=self.crop_bounds)
        return {"body_paths": body_file, "bodys": body, "cloth_paths": cloth_file, "input_cloths": source,
                "target_cloths": target}

import importlib

import torch

from datasets.base_dataset import BaseDataset


def find_dataset_using_name(name):
    """`--dataset foo_bar` -> class FooBarDataset (any case) in module datasets.foo_bar_dataset."""
    lib = importlib.import_module(f"datasets.{name}_dataset")
    want = name.replace("_", "") + "dataset"
    for key, cls in vars(lib).items():
        if key.lower() == want and isinstance(cls, type) and issubclass(cls, BaseDataset):
            return cls
    raise NotImplementedError(f"no dataset class for {name}")


def get_options_modifier(name):
    return find_dataset_using_name(name).modify_commandline_options


class CappedDataLoader:
    def __init__(self, opt):
        self.opt = opt
        self.dataset = find_dataset_using_name(opt.dataset or opt.model)(opt)
        print(f"dataset [{type(self.dataset).__name__}] was created")
        self.dataloader = torch.utils.data.DataLoader(self.dataset, batch_size=opt.batch_size, shuffle=False,
                                                      num_workers=opt.num_workers)

    def __len__(self):
        return min(len(self.dataset), self.opt.max_dataset_size)

    def __iter__(self):
        return iter(self.dataloader)


def create_dataset(opt):
    return CappedDataLoader(opt)

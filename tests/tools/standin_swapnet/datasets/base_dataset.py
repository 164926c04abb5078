import torch.utils.data


class BaseDataset(torch.utils.data.Dataset):
    def __init__(self, opt):
        self.opt = opt
        self.root = opt.dataroot
        self.is_train = opt.is_train
        self.crop_bounds = None
        if isinstance(opt.crop_size, int) and opt.crop_size < opt.load_size:   # centre crop, square
            lo = int((opt.load_size - opt.crop_size) / 2)
            self.crop_bounds = (lo, lo), (opt.load_size - lo, opt.load_size - lo)

    @staticmethod
    def modify_commandline_options(parser, is_train):
        return parser

import argparse

import datasets
import models


class TrainOptions:
    """Base + training flags, then the model's and the dataset's option modifiers, in one parser whose later
    definitions replace earlier ones (conflict_handler="resolve"), as the reference gathers its options.  The base
    --lr default (0.01) is the reference's: the model plugin must replace it.  The flags below the plugins' reach —
    weight_decay, init_type, b1/b2 (which the reference's optimizers package adds) — are this stand-in's own values,
    so a run against it checks the plugins' defaults only; SWAPNET_REFERENCE runs the same tests on the real parser."""

    def parse(self, print_options=True):
        p = argparse.ArgumentParser(conflict_handler="resolve")
        p.add_argument("--name", default="my_experiment")
        p.add_argument("--model", default="warp")
        p.add_argument("--dataset", default=None)
        p.add_argument("--dataroot", required=True)
        p.add_argument("--checkpoints_dir", default="./checkpoints")
        p.add_argument("--load_epoch", default="latest")
        p.add_argument("--dataset_mode", default="image")
        p.add_argument("--cloth_representation", default="labels")
        p.add_argument("--body_representation", default="rgb")
        p.add_argument("--cloth_channels", type=int, default=19)
        p.add_argument("--body_channels", type=int, default=12)
        p.add_argument("--texture_channels", type=int, default=3)
        p.add_argument("--load_size", type=int, default=128)
        p.add_argument("--crop_size", type=int, default=128)
        p.add_argument("--crop_bounds", default=None)
        p.add_argument("--max_dataset_size", type=int, default=float("inf"))
        p.add_argument("--batch_size", type=int, default=8)
        p.add_argument("--shuffle_data", type=bool, default=True)
        p.add_argument("--num_workers", type=int, default=4)
        p.add_argument("--gpu_id", type=int, default=0)
        p.add_argument("--no_confirm", action="store_true")
        p.add_argument("--verbose", action="store_true")
        p.add_argument("--display_id", type=int, default=1)
        p.add_argument("--display_ncols", type=int, default=4)
        p.add_argument("--n_epochs", type=int, default=20)
        p.add_argument("--continue_train", action="store_true")
        p.add_argument("--weight_decay", type=float, default=0)
        p.add_argument("--init_type", default="kaiming")
        p.add_argument("--init_gain", type=float, default=0.02)
        p.add_argument("--lr", type=float, default=0.01)
        p.add_argument("--b1", type=float, default=0.9)
        p.add_argument("--b2", type=float, default=0.999)
        known, _ = p.parse_known_args()
        p = models.get_options_modifier(known.model)(p, True)
        p = datasets.get_options_modifier(known.dataset or known.model)(p, True)
        opt = p.parse_args()
        opt.is_train = True
        if print_options:
            print("".join(f"{k}: {v}\n" for k, v in sorted(vars(opt).items())))
        return opt

"""Start-up of a training run as the reference's train.py does it: options, dataset, model."""
import models
from datasets import create_dataset
from options.train_options import TrainOptions

opt = TrainOptions().parse()
dataset = create_dataset(opt)
print(f"The number of training images = {len(dataset)}")
model = models.create_model(opt)
model.setup(opt)

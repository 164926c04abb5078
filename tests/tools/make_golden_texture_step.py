"""Generate tests/golden/texture_step_64.pt: ONE full reference `TextureModel.optimize_parameters()`
(models/texture_model.py:127-180, base_gan.py:194-203) with the reference's DEFAULT losses
(L1 10, GAN 1, VGG16 content 20, Gram style 1e-8), imported through oracle/ref_harness.py.

    SWAPNET_REFERENCE=/path/to/SwapNet python tests/tools/make_golden_texture_step.py

CPU (gpu_id=None), eval-mode nets (torch's dropout RNG cannot be restated), 64x64, batch 2.  `vgg16(pretrained=True)`
(modules/losses/perceptual.py:26) is patched to torchvision's seeded random init (see make_golden_perceptual.py).
The fixture holds the eight losses and checksums of every parameter after the D and G AdamW updates.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import torchvision

from oracle import ref_harness as RH

RH.import_reference()
import models as ref_models  # noqa: E402  (the reference's)
import modules.losses.perceptual as P  # noqa: E402

from test_engine_gpu import synth_texture_batch  # noqa: E402


def seeded(pretrained=False, **kw):
    with torch.random.fork_rng():
        torch.manual_seed(1234)
        return torchvision.models.vgg16(weights=None)


def checksums(sd):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()}


B, S = 2, 64
torch.manual_seed(0)
opt = RH.texture_opt(B, S, lambda_content=20.0, lambda_style=1e-8)
orig = P.vgg16
P.vgg16 = seeded
try:
    model = ref_models.create_model(opt)
finally:
    P.vgg16 = orig
model.setup(opt)
model.eval()
gold = dict(init_checksums_G=checksums(model.net_generator.state_dict()),
            init_checksums_D=checksums(model.net_discriminator.state_dict()))
tex, rois, cloth, tgt = synth_texture_batch(B, S)
torch.manual_seed(123)   # GANLoss draws its smooth labels from the CPU default generator
model.set_input(dict(input_textures=tex, rois=rois, cloths=cloth, target_textures=tgt, cloth_paths=["c"] * B,
                     texture_paths=["t"] * B))
model.optimize_parameters()
gold["step_losses"] = {k: float(v) for k, v in model.get_current_losses().items()}
gold["step_checksums_G"] = checksums(model.net_generator.state_dict())
gold["step_checksums_D"] = checksums(model.net_discriminator.state_dict())
torch.save(gold, os.path.join(ROOT, "tests", "golden", "texture_step_64.pt"))
print("texture_step_64.pt", gold["step_losses"])

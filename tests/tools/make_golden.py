"""Generate tests/golden/*.pt from the UNMODIFIED reference (oracle/ref_harness.py).

    SWAPNET_REFERENCE=/path/to/SwapNet python tests/tools/make_golden.py

Fixtures (all seeded; see tests/test_oracle_cpu.py for how they are consumed):
  warp_64.pt     reference WarpModule / define_D forward (eval) + one full reference
                 WarpModel.optimize_parameters() (eval-mode nets, CPU, gpu_id=None): six losses and
                 checksums of every updated parameter
  texture_64.pt  reference TextureModule forward (eval) at 64x64 incl. reshape_rois and the ROIAlign output
  roi_256.pt     torchvision RoIAlign on the notebook ROI fixture (256x256), strided subsample + sums
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

from oracle import ref_harness as RH
from oracle import roi_align as R

RH.import_reference()
import models as ref_models  # noqa: E402  (the reference's)
from modules import init_weights  # noqa: E402
from modules.swapnet_modules import TextureModule, WarpModule  # noqa: E402
from modules.discriminators import define_D  # noqa: E402

from test_engine_gpu import synth_texture_batch, synth_warp_batch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def checksums(sd):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()}


# ---- warp -------------------------------------------------------------------------------------
B, S = 1, 64
torch.manual_seed(0)
G = WarpModule(); init_weights(G, "kaiming")
D = define_D(22, 64, "basic", 3, "instance"); init_weights(D, "kaiming")
G.eval(); D.eval()
body, inp, tgt = synth_warp_batch(B, S)
with torch.no_grad():
    fakes = G(body, inp)
    pred = D(torch.cat((body, fakes), 1))
gold = dict(fakes=fakes, pred=pred, init_checksums_G=checksums(G.state_dict()), init_checksums_D=checksums(D.state_dict()))

torch.manual_seed(0)
opt = RH.warp_opt(B)
model = ref_models.create_model(opt)
model.setup(opt)
model.eval()            # dropout off (torch's dropout RNG cannot be restated); IN keeps no running stats
torch.manual_seed(123)  # GANLoss draws its smooth labels from the CPU default generator
model.set_input(dict(bodys=body, input_cloths=inp, target_cloths=tgt, cloth_paths=["c"], body_paths=["b"]))
model.optimize_parameters()
gold["step_losses"] = {k: float(v) for k, v in model.get_current_losses().items()}
gold["step_checksums_G"] = checksums(model.net_generator.state_dict())
gold["step_checksums_D"] = checksums(model.net_discriminator.state_dict())
gold["step_fakes"] = model.fakes.detach().clone()
torch.save(gold, os.path.join(OUT, "warp_64.pt"))
print("warp_64.pt", gold["step_losses"])

# ---- texture ------------------------------------------------------------------------------------
torch.manual_seed(0)
T = TextureModule(3, 19, 12, "instance", 0.5, "pix2pix", S); init_weights(T, "kaiming"); T.eval()
tex, rois, cloth, _ = synth_texture_batch(2, S)
with torch.no_grad():
    out = T(tex, rois, cloth.clone())
    r5 = TextureModule.reshape_rois(rois)
    pooled = T.roi_align(tex, r5).view(2, -1, 128, 128)
torch.save(dict(fakes=out, reshaped_rois=r5, pooled_sub=pooled[:, :, ::8, ::8].clone(),
                pooled_sum=pooled.double().sum((2, 3)), init_checksums=checksums(T.state_dict())),
           os.path.join(OUT, "texture_64.pt"))
print("texture_64.pt", tuple(out.shape))

# ---- ROIAlign on the notebook fixture -------------------------------------------------------------
from torchvision.ops import RoIAlign  # noqa: E402

S2 = 256
base = np.concatenate([R.NOTEBOOK_ROIS_256, R.NOTEBOOK_EXTRA_256])
rois_np = np.stack([np.roll(base, b, axis=0)[:12] for b in range(3)]).astype(np.float32)
rois_np[2, 5] = [-30, -20, 40, 50]
rois_np[1, 3] = [S2 + 5, S2 + 7, S2 + 40, S2 + 50]
rois_np[0, 7] = [10.5, 20.25, 11.0, 20.5]
texr = torch.randn(3, 3, S2, S2, generator=torch.Generator().manual_seed(0))
ra = RoIAlign(output_size=(128, 128), spatial_scale=1, sampling_ratio=1)
ref = ra(texr, TextureModule.reshape_rois(torch.from_numpy(rois_np))).view(3, -1, 128, 128)
torch.save(dict(rois=torch.from_numpy(rois_np), sub=ref[:, :, ::8, ::8].clone(), sums=ref.double().sum((2, 3))),
           os.path.join(OUT, "roi_256.pt"))
print("roi_256.pt", tuple(ref.shape))

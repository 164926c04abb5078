"""Generate tests/golden/perceptual_64.pt from the UNMODIFIED reference PerceptualLoss
(modules/losses/perceptual.py of the checkout oracle/ref_harness.py imports).

    SWAPNET_REFERENCE=/path/to/SwapNet python tests/tools/make_golden_perceptual.py

`vgg16(pretrained=True)` (perceptual.py:26) is a download and impossible offline: the constructor is patched
to torchvision's own seeded random init (torch.manual_seed(1234)), the same stand-in the B200 plugin uses with
`--b200_vgg random`.  The fixture holds the two loss values, a strided subsample and checksums of
d(20*content + 1e-8*style)/d(output), and checksums of the VGG weights (so that a different torchvision
initialisation would be noticed).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch
import torchvision

from oracle import ref_harness as RH

RH.import_reference()
import modules.losses.perceptual as P  # noqa: E402  (the reference's)


def seeded(pretrained=False, **kw):
    with torch.random.fork_rng():
        torch.manual_seed(1234)
        return torchvision.models.vgg16(weights=None)


orig = P.vgg16
P.vgg16 = seeded
try:
    crit = P.PerceptualLoss(use_style=True)
finally:
    P.vgg16 = orig
g = torch.Generator().manual_seed(5)
out = (torch.rand(2, 3, 64, 64, generator=g) * 2 - 1).requires_grad_()
tgt = torch.rand(2, 3, 64, 64, generator=g) * 4.5 - 2.0
c, s = crit(out, tgt)
(c * 20 + s * 1e-8).backward()
sd = seeded().features.state_dict()
gold = dict(content=float(c), style=float(s), grad_sub=out.grad[:, :, ::4, ::4].clone(),
            grad_sum=float(out.grad.double().sum()), grad_abs=float(out.grad.double().abs().sum()),
            vgg_checksums={k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()})
torch.save(gold, os.path.join(ROOT, "tests", "golden", "perceptual_64.pt"))
print("content", gold["content"], "style", gold["style"], "grad_abs", gold["grad_abs"])

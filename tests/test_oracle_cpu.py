"""Pins the CPU oracle (oracle/) against the reference: golden vectors generated from the UNMODIFIED
reference by tests/tools/make_golden*.py, committed under tests/golden/."""
import os

import numpy as np
import pytest
import torch

from oracle import dropout as OD
from oracle import nets as ON
from oracle import roi_align as R
from swapnet_b200 import modules as M
from test_engine_gpu import synth_texture_batch, synth_warp_batch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SUM_ORDER = 1e-13      # relative: float64 summation order (a different initialisation moves a checksum by > 1e-5)


def relmax(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


def checksums(sd):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()}


def close_checksums(a, b, tol, numel=None, lr=0.0):
    """flips / lr: checksums of parameters AFTER the first AdamW step.  That update is lr * g / (|g| + eps) ~ lr * sign(g),
    so an element whose gradient is within CPU-kernel rounding of zero (oneDNN picks different kernels on different
    hosts) moves by up to 2 * lr the other way; allow max(8, 2e-5 * numel) such elements per tensor on top of the
    relative bound (measured across two hosts: 9 of 8.4 M; a wrong gradient flips a large fraction).
    tol=0.0 still allows SUM_ORDER: the float64 sums of identical tensors differ in the last bits between hosts, whose
    CPU reductions add in different orders (measured: 2 ulp)."""
    assert a.keys() == b.keys()
    for k in a:
        for x, y in zip(a[k], b[k]):
            flips = 0 if numel is None else max(8, 2e-5 * numel[k])
            assert abs(x - y) <= max(tol, SUM_ORDER) * max(1.0, abs(y)) + 2 * lr * flips, (k, x, y)


def test_warp_forward_and_step_match_golden():
    g = torch.load(os.path.join(GOLD, "warp_64.pt"))
    torch.manual_seed(0)
    G = M.WarpModule(); M.init_weights(G, "kaiming")
    D = M.NLayerDiscriminator(22, 64, 3, "instance"); M.init_weights(D, "kaiming")
    # our parameter containers reproduce the reference's seeded init exactly
    close_checksums(checksums(G.state_dict()), g["init_checksums_G"], 0.0)
    close_checksums(checksums(D.state_dict()), g["init_checksums_D"], 0.0)
    body, inp, tgt = synth_warp_batch(1, 64)
    with torch.no_grad():
        fakes = ON.warp_forward(G.state_dict(), body, inp)
        pred = ON.patchgan_forward(D.state_dict(), torch.cat((body, fakes), 1))
    assert relmax(fakes, g["fakes"]) < 1e-5 and relmax(pred, g["pred"]) < 1e-5
    # one full optimize_parameters(): D step, then G step against the UPDATED discriminator
    sdG = {k: v.detach().clone().requires_grad_() for k, v in G.state_dict().items()}
    sdD = {k: v.detach().clone().requires_grad_() for k, v in D.state_dict().items()}
    optG = torch.optim.AdamW(list(sdG.values()), lr=1e-4, weight_decay=0, betas=(0.9, 0.999))
    optD = torch.optim.AdamW(list(sdD.values()), lr=4e-4, weight_decay=0.01, betas=(0.9, 0.999))
    torch.manual_seed(123)
    fk = ON.warp_forward(sdG, body, inp)
    t_fake, t_real = ON.smooth_label(torch.rand(1)), ON.smooth_label(torch.rand(1))
    lf = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, fk), 1).detach()), t_fake)
    lr = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, tgt), 1)), t_real)
    lD = 0.5 * (lf + lr)
    lD.backward()
    optD.step()
    ce = torch.nn.functional.cross_entropy(fk, torch.argmax(tgt, 1)) * 100
    gan = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, fk), 1)), ON.smooth_label(torch.rand(1)))
    (ce + gan).backward()
    optG.step()
    got = dict(D=lD.item(), D_real=lr.item(), D_fake=lf.item(), G=(ce + gan).item(), G_gan=gan.item(), G_ce=ce.item())
    for k, v in g["step_losses"].items():
        assert abs(got[k] - v) <= 1e-5 * abs(v), (k, got[k], v)
    close_checksums(checksums({k: v.detach() for k, v in sdG.items()}), g["step_checksums_G"], 2e-6, numel={k: v.numel() for k, v in sdG.items()}, lr=1e-4)
    close_checksums(checksums({k: v.detach() for k, v in sdD.items()}), g["step_checksums_D"], 2e-6, numel={k: v.numel() for k, v in sdD.items()}, lr=4e-4)


def test_texture_forward_matches_golden():
    g = torch.load(os.path.join(GOLD, "texture_64.pt"))
    torch.manual_seed(0)
    T = M.TextureModule(3, 19, 12, "instance", 0.5, 64); M.init_weights(T, "kaiming")
    close_checksums(checksums(T.state_dict()), g["init_checksums"], 0.0)
    tex, rois, cloth, _ = synth_texture_batch(2, 64)
    # ROI bookkeeping: bit-exact
    assert np.array_equal(R.reshape_rois(rois.numpy()), g["reshaped_rois"].numpy())
    pooled = R.roi_align_pack(tex.numpy(), rois.numpy(), 128)
    assert np.array_equal(pooled[:, :, ::8, ::8], g["pooled_sub"].numpy())
    with torch.no_grad():
        out = ON.texture_forward(T.state_dict(), tex, rois, cloth)
    assert relmax(out, g["fakes"]) < 1e-5


def test_roi_align_known_answer_notebook_fixture():
    """test/Test TextureDataset Draw ROIs.ipynb ROI tensor (incl. zero-area and out-of-bounds rows)."""
    g = torch.load(os.path.join(GOLD, "roi_256.pt"))
    tex = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(0))
    out = R.roi_align_pack(tex.numpy(), g["rois"].numpy(), 128)
    assert np.array_equal(out[:, :, ::8, ::8], g["sub"].numpy())
    assert np.allclose(out.astype(np.float64).sum((2, 3)), g["sums"].numpy(), rtol=0, atol=1e-9)


def test_roi_kernel_source_run_on_the_host_equals_torchvision_fixture(tmp_path):
    """csrc/roi_align.cu's device code compiled for the host (tests/tools/kernel_host_shim.py, g++ -ffp-contract=off):
    bit-identical to the torchvision fixture (notebook ROIs incl. zero-area, out-of-bounds and sub-pixel rows) and to the
    numpy oracle — the operation order of the kernel checked without a GPU (GPU run: test_roi_align_pack_bit_exact)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "tools"))
    import kernel_host_shim

    lib = kernel_host_shim.build_roi(str(tmp_path))
    if lib is None:
        pytest.skip("no g++")
    g = torch.load(os.path.join(GOLD, "roi_256.pt"))
    tex = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(0)).numpy()
    rois = np.ascontiguousarray(g["rois"].numpy(), dtype=np.float32)
    out = np.full((3, 128, 128, 36), -5, np.float32)                  # NHWC, channel = 3 * roi + rgb
    lib.run_roi(tex.ctypes.data, 3, 3, 256, 256, rois.ctypes.data, 12, 128, out.ctypes.data)
    got = out.transpose(0, 3, 1, 2)
    assert np.array_equal(got, R.roi_align_pack(tex, rois, 128))
    assert np.array_equal(got[:, :, ::8, ::8], g["sub"].numpy())


def test_dropout_restatement_is_deterministic_and_balanced():
    m = OD.keep_mask(77, 0.5, 1 << 16)
    assert np.array_equal(m, OD.keep_mask(77, 0.5, 1 << 16))
    assert 0.49 < m.mean() < 0.51
    assert not np.array_equal(m, OD.keep_mask(78, 0.5, 1 << 16))
    assert OD.keep_mask(5, 0.0, 1000).all()


def close_to_reference(got, ref, tol=1e-12):
    """`got` (float64) against a tests/golden/reference_modules.pt entry: the stored subsample element-wise and the
    checksums of the whole tensor, both within `tol` relative — float64 rounding, far below any difference of formula."""
    step = ref["shape"][-1] // ref["sub"].shape[-1]
    assert tuple(got.shape) == ref["shape"]
    assert relmax(got[..., ::step, ::step], ref["sub"]) < tol
    for x, y in zip((float(got.double().sum()), float(got.double().abs().sum())), ref["sums"]):
        assert abs(x - y) <= tol * abs(ref["sums"][1]), (x, y)


def test_oracle_is_bit_identical_to_reference_modules():
    """The oracle against the reference's WarpModule, define_D("basic") and TextureModule (pix2pix) in eval mode,
    stored by tests/tools/make_golden_reference.py.  Both sides run in float64: float32 results depend on the CPU
    kernels a host picks (~1e-5), float64 pins the arithmetic to 1e-12 on any host."""
    ref = torch.load(os.path.join(GOLD, "reference_modules.pt"))
    torch.manual_seed(0)
    G = M.WarpModule(); M.init_weights(G, "kaiming")
    D = M.NLayerDiscriminator(22, 64, 3, "instance"); M.init_weights(D, "kaiming")
    close_checksums(checksums(G.state_dict()), ref["warp_init"], 0.0)
    close_checksums(checksums(D.state_dict()), ref["disc_init"], 0.0)
    sdG = {k: v.double() for k, v in G.state_dict().items()}
    sdD = {k: v.double() for k, v in D.state_dict().items()}
    body, inp, _ = synth_warp_batch(2, 64)
    with torch.no_grad():
        fakes = ON.warp_forward(sdG, body.double(), inp.double())
        close_to_reference(fakes, ref["warp"])
        close_to_reference(ON.patchgan_forward(sdD, torch.cat((body.double(), fakes), 1)), ref["disc"])
    torch.manual_seed(0)
    T = M.TextureModule(3, 19, 12, "instance", 0.5, 128); M.init_weights(T, "kaiming")
    close_checksums(checksums(T.state_dict()), ref["texture_init"], 0.0)
    tex, rois, cloth, _ = synth_texture_batch(2, 128)
    with torch.no_grad():
        out = ON.texture_forward({k: v.double() for k, v in T.state_dict().items()}, tex.double(), rois.double(),
                                 cloth.double())
    close_to_reference(out, ref["texture"])
    # state_dict keys / seeded init of our containers == the reference's
    torch.manual_seed(3)
    b = M.WarpModule(); M.init_weights(b, "kaiming")
    assert list(b.state_dict()) == ref["seed3_keys"]
    close_checksums(checksums(b.state_dict()), ref["seed3_init"], 0.0)


def seeded_vgg_features_sd(seed=1234):
    """The stand-in for the unobtainable `vgg16(pretrained=True)`: torchvision's own constructor
    (kaiming_normal fan_out convs, zero bias) under a fixed seed (SURVEY App. C)."""
    import torchvision

    with torch.random.fork_rng():
        torch.manual_seed(seed)
        net = torchvision.models.vgg16(weights=None)
    return {k: v.detach().clone() for k, v in net.features.state_dict().items()}


def test_perceptual_oracle_is_bit_identical_to_reference():
    """The reference PerceptualLoss(use_style=True) with the seeded-random VGG16 (stored by
    tests/tools/make_golden_reference.py): both losses and d(20*content + 1e-8*style)/d(output), both sides in float64,
    within 1e-12 relative — float64 rounding, far below any difference of formula."""
    ref = torch.load(os.path.join(GOLD, "reference_modules.pt"))["perceptual"]
    sd = {k: v.double() for k, v in seeded_vgg_features_sd().items()}
    g = torch.Generator().manual_seed(5)
    out = torch.rand(2, 3, 64, 64, generator=g).double().requires_grad_()
    tgt = torch.rand(2, 3, 64, 64, generator=g).double()
    c, s_ = ON.perceptual_loss(sd, out, tgt, True)
    (c * 20 + s_ * 1e-8).backward()
    assert abs(c.item() - ref["content"]) <= 1e-12 * abs(ref["content"])
    assert abs(s_.item() - ref["style"]) <= 1e-12 * abs(ref["style"])
    close_to_reference(out.grad, ref["grad"])


def test_perceptual_oracle_matches_golden():
    """tests/golden/perceptual_64.pt: the reference PerceptualLoss(use_style=True) with seeded-random VGG16
    (generated by tests/tools/make_golden_perceptual.py) — pins the oracle where /root/reference is absent."""
    g = torch.load(os.path.join(GOLD, "perceptual_64.pt"))
    sd = seeded_vgg_features_sd()
    close_checksums({k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()},
                    g["vgg_checksums"], 1e-12)
    gen = torch.Generator().manual_seed(5)
    out = (torch.rand(2, 3, 64, 64, generator=gen) * 2 - 1).requires_grad_()
    tgt = torch.rand(2, 3, 64, 64, generator=gen) * 4.5 - 2.0
    c, s = ON.perceptual_loss(sd, out, tgt, True)
    (c * 20 + s * 1e-8).backward()
    assert abs(float(c) - g["content"]) <= 1e-6 * abs(g["content"])
    assert abs(float(s) - g["style"]) <= 1e-6 * abs(g["style"])
    assert relmax(out.grad[:, :, ::4, ::4], g["grad_sub"]) < 1e-5
    assert abs(float(out.grad.double().abs().sum()) - g["grad_abs"]) <= 1e-5 * g["grad_abs"]


def test_vgg16_container_and_loader():
    """swapnet_b200.modules.VGG16Features: torchvision key names, frozen, seeded 'random' init reproducible;
    'pretrained' must raise (no silent substitute) when the weight file cannot be obtained."""
    a = M.load_vgg16_features("random")
    b = M.load_vgg16_features("random:1234")
    c = M.load_vgg16_features("random:7")
    ref = seeded_vgg_features_sd(1234)
    assert list(a.state_dict()) == list(ref) and all(torch.equal(a.state_dict()[k], ref[k]) for k in ref)
    assert all(torch.equal(a.state_dict()[k], b.state_dict()[k]) for k in ref)
    assert not torch.equal(a.state_dict()["0.weight"], c.state_dict()["0.weight"])
    assert not any(p.requires_grad for p in a.parameters())
    hub = os.path.join(torch.hub.get_dir(), "checkpoints", "vgg16-397923af.pth")
    if not os.path.exists(hub):
        with pytest.raises(RuntimeError, match="b200_vgg"):
            M.load_vgg16_features("pretrained")


def test_texture_full_step_with_default_losses_matches_golden():
    """tests/golden/texture_step_64.pt: one full reference TextureModel.optimize_parameters() with the DEFAULT loss
    set (L1 10 + GAN 1 + VGG16 content 20 + Gram style 1e-8; seeded-random VGG16) — the oracle's
    texture_step_losses / perceptual_loss + AdamW must reproduce the eight losses and every updated parameter."""
    g = torch.load(os.path.join(GOLD, "texture_step_64.pt"))
    B, S = 2, 64
    torch.manual_seed(0)
    T = M.TextureModule(3, 19, 12, "instance", 0.5, S); M.init_weights(T, "kaiming")
    D = M.NLayerDiscriminator(22, 64, 3, "instance"); M.init_weights(D, "kaiming")
    close_checksums(checksums(T.state_dict()), g["init_checksums_G"], 0.0)
    close_checksums(checksums(D.state_dict()), g["init_checksums_D"], 0.0)
    vgg = seeded_vgg_features_sd()
    tex, rois, cloth, tgt = synth_texture_batch(B, S)
    sdG = {k: v.detach().clone().requires_grad_() for k, v in T.state_dict().items()}
    sdD = {k: v.detach().clone().requires_grad_() for k, v in D.state_dict().items()}
    optG = torch.optim.AdamW(list(sdG.values()), lr=1e-4, weight_decay=0, betas=(0.9, 0.999))
    optD = torch.optim.AdamW(list(sdD.values()), lr=4e-4, weight_decay=0.01, betas=(0.9, 0.999))
    torch.manual_seed(123)
    fk = ON.texture_forward(sdG, tex, rois, cloth)
    t_fake, t_real = ON.smooth_label(torch.rand(1)), ON.smooth_label(torch.rand(1))
    lf = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((cloth, fk), 1).detach()), t_fake)
    lr = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((cloth, tgt), 1)), t_real)
    lD = 0.5 * (lf + lr)
    lD.backward()
    optD.step()
    gan = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((cloth, fk), 1)), ON.smooth_label(torch.rand(1)))
    l1 = torch.nn.functional.l1_loss(fk, tgt) * 10
    c, s_ = ON.perceptual_loss(vgg, fk, tgt, True)
    lG = gan + l1 + c * 20 + s_ * 1e-8
    lG.backward()
    optG.step()
    got = dict(D=lD.item(), D_real=lr.item(), D_fake=lf.item(), G=lG.item(), G_gan=gan.item(), G_l1=l1.item(),
               G_content=(c * 20).item(), G_style=(s_ * 1e-8).item())
    for k, v in g["step_losses"].items():
        assert abs(got[k] - v) <= 2e-5 * abs(v), (k, got[k], v)
    close_checksums(checksums({k: v.detach() for k, v in sdG.items()}), g["step_checksums_G"], 5e-6, numel={k: v.numel() for k, v in sdG.items()}, lr=1e-4)
    close_checksums(checksums({k: v.detach() for k, v in sdD.items()}), g["step_checksums_D"], 5e-6, numel={k: v.numel() for k, v in sdD.items()}, lr=4e-4)


@pytest.mark.parametrize("B", [1, 2])
def test_imposed_gates_do_not_change_the_oracle_gradient(B):
    """Imposing the gates the oracle would choose itself — delivered the way the GPU tests deliver the device's gates,
    as a permuted NHWC view — must leave every gradient unchanged.  (Regression: with a channels-last-strided mask
    torch.where returns a channels-last tensor and torch's CPU instance_norm backward returns a wrong gradient for batch
    size 1; oracle/nets.py:_act makes the mask contiguous.  This cost the 512x512 batch-1 step tests a day.)"""
    torch.manual_seed(0)
    G = M.WarpModule(); M.init_weights(G, "kaiming")
    body, inp, _ = synth_warp_batch(B, 64)
    grads = {}
    for mode in ("plain", "gated"):
        sd = {k: v.detach().double().requires_grad_() for k, v in G.state_dict().items()}
        if mode == "gated":
            ON.gate_with(lambda name, x: (x.detach() > 0).permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2))
        out = ON.warp_forward(sd, body.double(), inp.double())
        ON.gate_with(None)
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(5)).double()
        grads[mode] = torch.autograd.grad(out, list(sd.values()), g, allow_unused=True)
    for (k, _), a, b in zip(G.state_dict().items(), grads["plain"], grads["gated"]):
        if a is not None:
            assert torch.equal(a, b), k

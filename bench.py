#!/usr/bin/env python
"""SwapNet GAN-training throughput on B200 (BASELINE.json metric: images/s of the full G+D training step).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (default: warp stage, configs[1])
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (baseline arm, same config object)
    torchrun --nproc-per-node N bench.py --gpus N ...        # data parallel, one rank per GPU (NCCL)
    python bench.py --model texture --perceptual             # BASELINE configs[2] (default texture losses incl. VGG16)
    python bench.py --model joint --perceptual               # configs[4]: one warp + one texture step, 8 images/GPU
    python bench.py --device-augment                         # e2e leg with the dataset's augmentation on the device (f4)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write what the last timed step computed, DIR/*.npy

One "step" = one `optimize_parameters()` of the plugin (G fwd, D step on fake+real, G step through D, both AdamW updates —
the full reference training step, models/warp_model.py:169-183 / texture_model.py:127-180) on a synthetic batch of
`--batch` 512x512 images per GPU (default 16).  stdout carries exactly ONE JSON line (rank 0); everything else that
libraries print (NCCL banner ...) is routed to stderr.  Field notes:
  value     images/s, whole job, inputs already resident in HBM, K steps between CUDA events after W >= 3 warm-up steps
            (the step is replayed as a CUDA graph from the third step of a shape on; multi-GPU steps launch eagerly);
  e2e       same metric through set_input / optimize_parameters / get_current_losses (train.py:62-74) with PINNED HOST
            tensors: every step's H2D copy and the one 64-byte D2H of the losses are inside the timed region.  The cloth
            tensors travel as uint8 label maps (ops.SegMap, expanded on the device) unless --fp32-inputs (the 19-channel
            fp32 tensors the reference's DataLoader yields: 688 MB per batch-16 step); --device-augment ships one label
            map per sample + the drawn op table and runs the per-channel augmentation on the device inside the region;
  roofline  dominant kernel class = the tcgen05 tap-GEMM (`tap_gemm_kernel<3>`: forward + dgrad launches): algorithmic
            conv FLOPs of those launches / their summed CUDA-event time in one extra eager step, against the measured
            sustained dense bf16 peak (MEASURED_PEAKS.json).  The kernel issues 3 MMAs per algorithmic MAC (fp16/bf16-split
            fp32-faithful product), so frac <= 1/3 by construction; `pipe_frac` is the tensor-pipe view (3x);
            `resblock` = the eight resblock convs alone (fwd / dgrad / wgrad), `wgrad_kernel` = all weight gradients;
            `traffic` = DRAM bytes per launch from the committed ncu capture (a constant from profiles/, not measured here);
  cpu_baseline  the CPU oracle port (oracle/nets.py, pinned bit-exactly to the reference modules) running the same
            training step at 512x512, batch 1, on the host cores the cgroup quota allows (host_cores()), `--cpu-steps`
            steps (N = 1 only; --no-cpu-baseline skips it);
  --impl reference   the same port as the reference arm: exactly K timed and W warm-up steps, each on `--cpu-batch`
            image(s) of the batch (a bounded sample: the step is per-sample work + batch-mean losses), same `config`.
            The reference is pure Python: there is nothing to compile into oracle/_ref, so `kind` is "port"; where
            SWAPNET_REFERENCE names a checkout of the reference the warp arm times the UNMODIFIED reference WarpModel
            through its own API instead (`kind` "reference").
  --dump-outputs DIR  after the timed steps, what the last of them returned to its caller, one float array per file:
            <stage>_loss_<name>.npy (float64 scalars of get_current_losses()) and <stage>_fakes.npy (float32, the
            generator's output; above DUMP_ELEMENTS elements a fixed seeded sample of its flattened elements, the same
            positions on every run).  Inputs and weights are seeded, so two builds can be compared file by file —
            with a tolerance: the kernels accumulate with float atomics, and AdamW amplifies the rounding differences
            from step to step (two runs of one build, warp, 13 steps at 512x512 batch 16 on a B200 at 1000 W: losses
            within 1e-5 relative, fakes within 5e-2).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FULL_STEP_GFLOP_PER_IMG_512 = 1029.0   # SURVEY §8(d): full reference warp training step, nominal
DUMP_ELEMENTS = 1 << 22                # per dumped array: 16 MB of float32, so a joint run stays under 64 MB in all


def step_gflop_per_img(args) -> float:
    """Nominal conv GFLOP of one training step per 512x512 image (SURVEY §8d table)."""
    tex = 896.0 if args.perceptual else 415.0
    return {"warp": FULL_STEP_GFLOP_PER_IMG_512, "texture": tex, "joint": FULL_STEP_GFLOP_PER_IMG_512 + tex}[args.model]


def metric_name(args) -> str:
    return {"warp": "images/sec (G+D fwd+bwd) warp-stage 512x512",
            "texture": "images/sec (G+D fwd+bwd) texture-stage 512x512",
            "joint": "images/sec (G+D fwd+bwd) joint warp+texture 512x512"}[args.model]


def synth_batch(B, S, seed, labels=False):
    """SURVEY §8(d): normalised-RGB-like body, 16x16-block one-hot cloth (label 0 = all-zero),
    input cloth = target rolled by (8, 8).  labels=True: the two cloth tensors in compact form — uint8 label maps
    [B,S,S], the wire format the plugin expands on the device (ops.SegMap) — instead of fp32 one-hot [B,19,S,S]."""
    g = torch.Generator().manual_seed(seed)
    body = torch.rand(B, 3, S, S, generator=g) * 4.8 - 0.31
    lab = torch.randint(0, 19, (B, S // 16, S // 16), generator=g).repeat_interleave(16, 1).repeat_interleave(16, 2)
    if labels:
        lab = lab.to(torch.uint8)
        return dict(bodys=body, input_cloths=torch.roll(lab, (8, 8), (1, 2)).contiguous(), target_cloths=lab.contiguous(),
                    cloth_paths=["synthetic"] * B, body_paths=["synthetic"] * B)
    tgt = torch.zeros(B, 19, S, S)
    for c in range(1, 19):
        tgt[:, c] = (lab == c).float()
    inp = torch.roll(tgt, (8, 8), (2, 3))
    return dict(bodys=body, input_cloths=inp, target_cloths=tgt, cloth_paths=["synthetic"] * B,
                body_paths=["synthetic"] * B)


def synth_texture_batch(B, S, seed, labels=False):
    """SURVEY §8(d) config 3: normalised-RGB-like textures, one-hot cloth, rois = notebook fixture (256 px
    space, incl. degenerate rows) scaled to S and rotated per sample.  labels=True: the cloth tensor as a uint8 label
    map [B,S,S] (expanded on the device) instead of fp32 one-hot [B,19,S,S]."""
    g = torch.Generator().manual_seed(seed)
    tex = torch.rand(B, 3, S, S, generator=g) * 4.5 - 2.0
    tgt = torch.rand(B, 3, S, S, generator=g) * 4.5 - 2.0
    lab = torch.randint(0, 19, (B, S // 16, S // 16), generator=g).repeat_interleave(16, 1).repeat_interleave(16, 2)
    if labels:
        cloth = lab.to(torch.uint8).contiguous()
    else:
        cloth = torch.zeros(B, 19, S, S)
        for c in range(1, 19):
            cloth[:, c] = (lab == c).float()
    base = torch.tensor([[159, 0, 193, 14], [144, 15, 206, 89], [255, 0, 255, 0], [196, 20, 215, 94],
                         [144, 151, 180, 229], [179, 151, 216, 226], [156, 1, 188, 24], [141, 83, 215, 155],
                         [128, 20, 160, 82], [206, 92, 226, 158], [145, 220, 168, 255], [174, 217, 203, 255]],
                        dtype=torch.float32) * (S / 256.0)
    rois = torch.stack([torch.roll(base, b, 0) for b in range(B)])
    return dict(input_textures=tex, rois=rois, cloths=cloth, target_textures=tgt, cloth_paths=["synthetic"] * B,
                texture_paths=["synthetic"] * B)


class device_augment_feed:
    """SURVEY §8 f4 as a bench leg: what a DataLoader built on swapnet_b200/data.py hands over per step — the body
    images (fp32, pinned), ONE uint8 label map per sample (in the reference's image mode the input cloth is the target
    cloth before augmentation, datasets/warp_dataset.py:98-100) and the op table of the per-channel augmentation
    (drawn here once, before the timed region, with the reference's transform set; the reference draws in its DataLoader
    workers too).  Calling it does the H2D copies and the augmentation on the device and returns the `set_input` dict."""

    def __init__(self, B, S, seed):
        import random

        from torchvision import transforms as T

        from swapnet_b200 import data as D

        base = synth_batch(B, S, seed, labels=True)
        self.body, self.labels = base["bodys"].pin_memory(), base["target_cloths"].pin_memory()
        tf = T.RandomOrder([T.RandomVerticalFlip(), T.RandomHorizontalFlip(),        # datasets/__init__.py:88-110
                            T.RandomAffine(degrees=10, translate=(0.1, 0.1), scale=(0.8, 1.2), shear=20),
                            T.RandomPerspective()])
        self.aug = D.ClothAugmenter(tf, 19)
        py_state = random.getstate()
        with torch.random.fork_rng(devices=[]):          # the plugin's smooth-label draws use the global CPU generator
            random.seed(seed)
            torch.manual_seed(seed)
            t0 = time.perf_counter()
            self.table = D.OpTable([self.aug.draw(S, S) for _ in range(B)])
            self.draw_ms_per_sample = (time.perf_counter() - t0) * 1e3 / B
        random.setstate(py_state)
        self.B = B
        self.h2d_bytes = (self.body.numel() * 4 + self.labels.numel() + self.table.nbytes)

    def __call__(self):
        from swapnet_b200.ops import SegMap

        lab = self.labels.cuda(non_blocking=True)
        return dict(bodys=self.body, input_cloths=self.aug.apply(lab, self.table), target_cloths=SegMap(lab, 19),
                    cloth_paths=["synthetic"] * self.B, body_paths=["synthetic"] * self.B)

    def resident(self):
        d = self()
        d["bodys"] = self.body.cuda()
        return d


def warp_opt(B, S, precision):
    return argparse.Namespace(
        model="warp", gpu_id=int(os.environ.get("LOCAL_RANK", 0)), is_train=True,
        checkpoints_dir=tempfile.mkdtemp(prefix="sn_bench_"), name="warp", no_confirm=True,
        body_representation="rgb", body_channels=12, cloth_representation="labels", cloth_channels=19,
        texture_channels=3, init_type="kaiming", init_gain=0.02, discriminator="basic", n_layers_D=3,
        norm="instance", gan_mode="vanilla", gan_label_mode="smooth", lambda_gan=1.0, lambda_discriminator=1.0,
        lambda_gp=10, optimizer_G="AdamW", optimizer_D="AdamW", lr=1e-4, d_lr=4e-4, weight_decay=0,
        d_weight_decay=0.01, b1=0.9, b2=0.999, warp_mode="gan", lambda_ce=100, continue_train=False,
        load_epoch="latest", verbose=False, batch_size=B, crop_size=S, load_size=S, b200_precision=precision)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.rows.append(f)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def ncu_traffic():
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/r02_ncu_traffic.json); null if absent."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            return json.load(open(p))
    return None


def dump_outputs(models, out_dir) -> None:
    """--dump-outputs: the losses and generator output of each model's most recent step (see the module docstring)."""
    os.makedirs(out_dir, exist_ok=True)
    for m in models:
        for name, v in m.get_current_losses().items():
            np.save(os.path.join(out_dir, f"{m.opt.model}_loss_{name}.npy"), np.float64(v))
        fakes = m.fakes.detach().float().contiguous().cpu().numpy().ravel()
        if fakes.size > DUMP_ELEMENTS:
            fakes = fakes[np.unique(np.random.default_rng(0).integers(0, fakes.size, DUMP_ELEMENTS))]
        np.save(os.path.join(out_dir, f"{m.opt.model}_fakes.npy"), fakes)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference training step restated in oracle/nets.py (bit-identical to the reference
# modules), with torch.optim.AdamW as optimizers/__init__.py builds it
# ------------------------------------------------------------------------------------------------
def host_cores() -> int:
    """CPUs this process may actually use: the scheduler affinity capped by the cgroup CPU quota (the GPU boxes
    expose 128 logical CPUs under a 16-CPU quota — 128 torch threads there are 8x oversubscribed)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]          # cgroup v2
        if q != "max":
            quota = int(q) / int(p)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())      # cgroup v1
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota is not None:
        n = min(n, max(1, int(quota + 0.999)))
    return max(1, n)


def cpu_unmodified_reference_run(S, B, steps, warmup):
    """The UNMODIFIED reference `WarpModel` (models/warp_model.py, imported from the checkout SWAPNET_REFERENCE names
    through oracle/ref_harness.py) timed through its own public API — set_input / optimize_parameters / get_current_losses, the
    calls of train.py:62-74 — on the host cores.  Without that checkout the arm takes the port
    (`cpu_reference_run`).  -> (images/s, median s) or None."""
    from oracle import ref_harness as RH

    if not RH.available() or os.environ.get("SN_BENCH_PORT") == "1":     # SN_BENCH_PORT=1: time the port (A/B)
        return None
    import contextlib

    torch.set_num_threads(host_cores())
    with contextlib.redirect_stdout(sys.stderr):
        try:
            RH.import_reference()
        except RuntimeError:            # this repo's `models` plugin is already imported in this process
            return None
        import models as ref_models

        torch.manual_seed(0)
        model = ref_models.create_model(RH.warp_opt(B, crop_size=S, load_size=S))
        model.setup(model.opt)
    batch = synth_batch(B, S, 1234)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        model.set_input(batch)
        model.optimize_parameters()
        model.get_current_losses()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return B / med, med


def cpu_reference_run(S, B, steps, warmup, model="warp", perceptual=False):
    """K timed steps (after W warm-up steps) of the reference training step on the host cores -> (images/s, median s).
    model: warp | texture | joint (one warp step + one texture step per iteration, BASELINE configs[4])."""
    from oracle import nets as ON
    from swapnet_b200 import modules as M

    import contextlib

    torch.set_num_threads(host_cores())
    g = torch.Generator().manual_seed(7)

    def drop(name, x):  # training-mode dropout(0.5) as in the reference (cost parity; masks irrelevant)
        return torch.nn.functional.dropout(x, 0.5, True)

    def leaf(net):
        return {k: v.detach().clone().requires_grad_() for k, v in net.state_dict().items()}

    def adamw(sd, lr, wd):
        return torch.optim.AdamW(list(sd.values()), lr=lr, weight_decay=wd, betas=(0.9, 0.999))

    steps_fns = []
    torch.manual_seed(0)
    if model in ("warp", "joint"):
        with contextlib.redirect_stdout(sys.stderr):
            G = M.WarpModule()
            M.init_weights(G, "kaiming")
            D = M.NLayerDiscriminator(22, 64, 3, "instance")
            M.init_weights(D, "kaiming")
        sdG, sdD = leaf(G), leaf(D)
        optG, optD = adamw(sdG, 1e-4, 0), adamw(sdD, 4e-4, 0.01)
        b = synth_batch(B, S, 1234)
        body, inp, tgt = b["bodys"], b["input_cloths"], b["target_cloths"]

        def warp_step():
            fakes = ON.warp_forward(sdG, body, inp, drop)
            optD.zero_grad()
            t = [ON.smooth_label(torch.rand(1, generator=g)) for _ in range(3)]
            lf = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, fakes), 1).detach()), t[0])
            lr = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, tgt), 1)), t[1])
            (0.5 * (lf + lr)).backward()
            optD.step()
            optG.zero_grad()
            ce = torch.nn.functional.cross_entropy(fakes, torch.argmax(tgt, 1)) * 100
            gan = ON.gan_loss(ON.patchgan_forward(sdD, torch.cat((body, fakes), 1)), t[2])
            (ce + gan).backward()
            optG.step()

        steps_fns.append(warp_step)
    if model in ("texture", "joint"):
        with contextlib.redirect_stdout(sys.stderr):
            T = M.TextureModule(3, 19, 12, "instance", 0.5, S)
            M.init_weights(T, "kaiming")
            DT = M.NLayerDiscriminator(22, 64, 3, "instance")
            M.init_weights(DT, "kaiming")
            vgg = None
            if perceptual:
                vgg = {k: v.detach() for k, v in M.load_vgg16_features("random").state_dict().items()}
        sdT, sdDT = leaf(T), leaf(DT)
        optT, optDT = adamw(sdT, 1e-4, 0), adamw(sdDT, 4e-4, 0.01)
        tb = synth_texture_batch(B, S, 1234)
        lc, ls = (20.0, 1e-8) if perceptual else (0.0, 0.0)

        def texture_step():
            draws = [torch.rand(1, generator=g) for _ in range(3)]
            o = ON.texture_step_losses(sdT, sdDT, tb["input_textures"], tb["rois"], tb["cloths"], tb["target_textures"],
                                       draws, drop=drop, vgg=vgg, lambda_content=lc, lambda_style=ls)
            optDT.zero_grad()
            o["D"].backward(retain_graph=True)
            optDT.step()
            optT.zero_grad()
            o["G"].backward()        # (evaluates D once for both phases: slightly LESS work than the reference)
            optT.step()

        steps_fns.append(texture_step)

    def step():
        for f in steps_fns:
            f()

    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return B / med, med


_REAL_STDOUT = None


def _protect_stdout():
    """stdout carries exactly ONE JSON line: everything else written to fd 1 from here on — Python prints, but also
    C-level writes such as NCCL's version banner — goes to stderr; emit() writes to the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj) -> None:
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default 16; 8 for --model joint)")
    ap.add_argument("--cpu-batch", type=int, default=1,
                    help="--impl reference: images per CPU step (a bounded sample of the batch)")
    ap.add_argument("--fp32-inputs", dest="labels", action="store_false",
                    help="feed the warp cloth tensors as the fp32 one-hot [B,19,S,S] tensors the reference's DataLoader "
                         "yields (688 MB of H2D per step at batch 16) instead of uint8 label maps expanded on the device "
                         "(the default: ops.SegMap, SURVEY 8f rank 4)")
    ap.add_argument("--device-augment", action="store_true",
                    help="warp: the e2e leg ships ONE uint8 label map per sample + the drawn op table and runs the reference's "
                         "per-channel augmentation (datasets/data_utils.py:346-361, --input_transforms hflip vflip affine "
                         "perspective) on the device (swapnet_b200/data.py) inside the timed region")
    ap.add_argument("--precision", default="fp32x3", choices=("fp32x3", "bf16"))
    ap.add_argument("--cpu-steps", type=int, default=3,
                    help="timed CPU-oracle steps of the cpu_baseline leg (one step = ~5 s on the usable host cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--perceptual", action="store_true",
                    help="--model texture: add the VGG16 content + Gram style terms (lambda 20 / 1e-8)")
    ap.add_argument("--model", default="warp", choices=("warp", "texture", "joint"),
                    help="warp = the BASELINE.json metric (default); texture = configs[2]; joint = configs[4] "
                         "(one warp step + one texture step per iteration)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the losses and the generator output of the last one as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the timed CUDA path computed: --impl b200 only")
    _protect_stdout()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    S = args.size
    B = args.batch if args.batch else (8 if args.model == "joint" else 16)   # BASELINE configs[1,2]: 16/GPU; [4]: 8/GPU
    cores = host_cores()
    tex_losses = ("L1 + GAN + VGG16 content + Gram style, seeded-random VGG weights" if args.perceptual
                  else "L1 + GAN; perceptual terms off")
    workload = {
        "warp": f"warp_model {S}x{S} synthetic, batch {B}/GPU, full GAN step (G fwd, D step, G step, AdamW x2)",
        "texture": f"texture_model {S}x{S} synthetic, 12-ROI, batch {B}/GPU, full GAN step ({tex_losses})",
        "joint": f"joint warp+texture {S}x{S} synthetic, batch {B}/GPU, one full warp GAN step + one full texture GAN step "
                 f"per iteration ({tex_losses})"}[args.model]
    config = {"workload": workload, "global_batch": B * world, "parallelism": f"dp{world}",
              "l2": "inputs+activations per step (>2 GB) exceed the 126 MB L2; no explicit flush",
              "algorithmic_tflop_per_step": step_gflop_per_img(args) * (S / 512) ** 2 * B * world / 1e3}

    if args.impl == "reference":
        if rank != 0:
            return
        # exactly K timed and W warm-up steps of the same workload and config; each CPU step is a BOUNDED SAMPLE of the
        # batch (`--cpu-batch` images, default 1: the step is per-sample work + batch-mean losses, cost linear in the
        # batch) so that 25 steps stay within a few minutes on the box's host cores
        unmodified = cpu_unmodified_reference_run(S, args.cpu_batch, args.steps, args.warmup) if args.model == "warp" else None
        if unmodified is not None:
            v, med = unmodified
            emit({"impl": "reference", "metric": metric_name(args), "value": v, "unit": "images/s", "n_gpus": args.gpus,
                  "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
                  "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                  "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "reference",
                                   "sample": f"{args.steps} timed + {args.warmup} warm-up steps of the UNMODIFIED reference "
                                             f"WarpModel (set_input + optimize_parameters + get_current_losses) at {S}x{S}, "
                                             f"each on {args.cpu_batch} image(s) of the batch, torch CPU fp32, {cores} threads"},
                  "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
            return
        v, med = cpu_reference_run(S, args.cpu_batch, args.steps, args.warmup, args.model, args.perceptual)
        emit(({
            "impl": "reference", "metric": metric_name(args), "value": v,
            "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} timed + {args.warmup} warm-up full training steps at {S}x{S}, each on "
                                       f"{args.cpu_batch} image(s) of the batch (bounded sample), torch CPU fp32 "
                                       f"({cores} threads = usable host cores); oracle/nets.py, pinned bit-exactly to the "
                                       "reference modules (the reference is pure Python: nothing to compile into oracle/_ref)"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback of the hot path)")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_MAX_CTAS", "16")     # see swapnet_b200/parallel.py:init_from_env
        torch.distributed.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    from swapnet_b200 import ops
    from swapnet_b200.models import create_model

    torch.manual_seed(0)
    import contextlib

    def texture_opt():
        o = warp_opt(B, S, args.precision)
        o.model, o.name, o.netG, o.lambda_l1, o.lambda_content, o.lambda_style = "texture", "texture", "swapnet", 10, 0, 0
        if args.perceptual:   # the reference's default texture losses; seeded-random VGG16 (no weight file offline)
            o.lambda_content, o.lambda_style, o.b200_vgg = 20.0, 1e-8, "random"
        return o

    # legs = [(model, pinned host batch, device-resident batch)]: one per stage (joint = warp then texture)
    legs = []
    with contextlib.redirect_stdout(sys.stderr):   # stdout carries exactly one JSON line
        for kind in (("warp", "texture") if args.model == "joint" else (args.model,)):
            o = warp_opt(B, S, args.precision) if kind == "warp" else texture_opt()
            m = create_model(o)
            m.setup(m.opt)
            if kind == "warp" and args.device_augment:
                host, tkeys = device_augment_feed(B, S, 1234 + rank), ("bodys", "input_cloths", "target_cloths")
                devb = host.resident()
                legs.append((m, host, devb, tkeys))
                continue
            if kind == "warp":
                host = synth_batch(B, S, 1234 + rank, labels=args.labels)
                tkeys = ("bodys", "input_cloths", "target_cloths")
            else:
                host = synth_texture_batch(B, S, 1234 + rank, labels=args.labels)
                tkeys = ("input_textures", "rois", "cloths", "target_textures")
            for k in tkeys:
                host[k] = host[k].pin_memory()
            devb = dict(host)
            for k in tkeys:
                devb[k] = host[k].cuda(non_blocking=True)
            legs.append((m, host, devb, tkeys))
    h2d = sum(host.h2d_bytes if callable(host) else sum(host[k].numel() * host[k].element_size() for k in tkeys)
              for _, host, _, tkeys in legs)
    n_losses = sum(len([n for n in m.loss_names if isinstance(n, str)]) for m, *_ in legs)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def one_step(on_host, read_losses):
        for m, host, devb, _ in legs:
            m.set_input((host() if callable(host) else host) if on_host else devb)
            m.optimize_parameters()
            if read_losses:
                m.get_current_losses()

    def timed(n, on_host, read_losses):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            one_step(on_host, read_losses)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item()

    for _ in range(max(args.warmup, 3)):
        one_step(False, False)
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ops.launch_count()
    ms = timed(args.steps, False, False)
    launches = ops.launch_count() - l0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:     # before the e2e leg's steps move the weights on
        dump_outputs([m for m, *_ in legs], args.dump_outputs)
    for _ in range(2):                      # the host-input path has its own staging buffers: warm them
        one_step(True, True)
    ms_e2e = timed(args.steps, True, True)

    # ---- roofline pass (untimed): per-launch CUDA events on the GEMM plans ----
    roof = None
    # every rank runs the traced step (it contains the gradient all-reduces); rank 0 evaluates it
    ops.Plan.trace = []
    for m, *_ in legs:
        m.graph_enabled = False             # per-launch events need eager launches
    one_step(False, False)
    torch.cuda.synchronize()
    trace, ops.Plan.trace = ops.Plan.trace, None
    if rank == 0:
        info = {}
        for m, *_ in legs:
            engs = [m._eng_G, m._eng_Dd, m._eng_Dg]
            pe = getattr(m, "_eng_P", None)
            if pe is not None and pe.out is not None:
                engs += [pe.out, pe.tgt]
            for eng in engs:
                for st in eng.stages:
                    fl, ly = 2.0 * st.nominal_macs(), st.layer
                    for p in ly.fwd_plans:
                        info[id(p)] = ("fwd", fl / len(ly.fwd_plans), st.name)
                    for p in ly.dgrad_plans:
                        info[id(p)] = ("dgrad", fl / len(ly.dgrad_plans), st.name)
                    if ly.wgrad_plan is not None:
                        info[id(ly.wgrad_plan)] = ("wgrad", fl, st.name)
        peak, hbm, how = measured_peaks()
        tot = {k: [0.0, 0.0, 0] for k in ("fwd", "dgrad", "wgrad", "res_fwd", "res_dgrad", "res_wgrad")}  # flops, ms, n
        for plan, a, b_ in trace:
            kind, fl, name = info[id(plan)]
            dt = a.elapsed_time(b_)
            for key in ((kind, "res_" + kind) if name.startswith("resblocks.") else (kind,)):
                tot[key][0] += fl
                tot[key][1] += dt
                tot[key][2] += 1
        gemm_fl = tot["fwd"][0] + tot["dgrad"][0]
        gemm_ms = tot["fwd"][1] + tot["dgrad"][1]
        gemm_n = tot["fwd"][2] + tot["dgrad"][2]
        step_ms = ms / args.steps

        def tf(key):
            return (tot[key][0] / (tot[key][1] * 1e-3) / 1e12) if tot[key][1] else 0.0

        ach = gemm_fl / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        res_fl = tot["res_fwd"][0] + tot["res_dgrad"][0]
        res_ms = tot["res_fwd"][1] + tot["res_dgrad"][1]
        res = (res_fl / (res_ms * 1e-3) / 1e12) if res_ms else 0.0
        tr = ncu_traffic()
        roof = {"bound": "tensor", "kernel": "tap_gemm_kernel<3> (tcgen05, fwd+dgrad launches)", "achieved": ach,
                "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "pipe_frac": 3 * ach / peak, "peak_source": how,
                "launches_per_step": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                "algorithmic_gflop_per_launch": gemm_fl / max(gemm_n, 1) / 1e9,
                "share_of_step": gemm_ms / step_ms,
                # DRAM bytes of one launch of the dominant shape: a constant from the committed `ncu --set full`
                # capture (profiles/), NOT measured in this run
                "traffic": (tr or {}).get("dram_bytes_per_launch"), "traffic_source": "committed ncu capture (profiles/)",
                "traffic_detail": tr,
                # the fused U-Net conv blocks the north-star target is read against: the 8 resblock convs
                # (59 % of generator FLOPs), FLOP-weighted over their fwd + dgrad launches, and their wgrad launches
                "resblock": {"achieved": res, "frac": res / peak, "pipe_frac": 3 * res / peak,
                             "launches_per_step": tot["res_fwd"][2] + tot["res_dgrad"][2],
                             "fwd": tf("res_fwd"), "dgrad": tf("res_dgrad"), "wgrad": tf("res_wgrad")},
                "wgrad_kernel": {"achieved": tf("wgrad"), "frac": tf("wgrad") / peak,
                                 "share_of_step": tot["wgrad"][1] / step_ms, "launches_per_step": tot["wgrad"][2]}}

    if rank != 0:
        torch.distributed.destroy_process_group()
        return
    cpu = None
    if not args.no_cpu_baseline and args.gpus == 1:
        v, med = cpu_reference_run(S, 1, args.cpu_steps, 1, args.model, args.perceptual)
        cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
               "sample": f"{args.cpu_steps} timed full training step(s) at {S}x{S}, batch 1, after 1 warm-up step, "
                         f"torch CPU ({cores} threads = usable cores under the cgroup quota)"}
    step_ms = ms / args.steps
    total_imgs = B * world
    out = {
        "metric": metric_name(args),
        "value": total_imgs / (step_ms * 1e-3),
        "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16/bf16-split x3 tensor-core products, fp32 accumulate (fp32-faithful)" if args.precision == "fp32x3"
        else "fp16 single-pass tensor-core products, fp32 accumulate",
        "data": "synthetic", "config": config,
        "e2e": {"value": total_imgs / (ms_e2e / args.steps * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": n_losses * 8,
                "inputs": ("ONE uint8 label map per sample + the op table of the reference's per-channel augmentation "
                           "(hflip, vflip, affine, perspective; draws made beforehand on the host), augmented and expanded "
                           "on the device inside the timed region (swapnet_b200/data.py)") if args.device_augment else
                "uint8 label maps for the cloth tensors (ops.SegMap), expanded to one-hot planes on the device"
                if args.labels else "fp32 tensors as the reference's DataLoader yields them"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
    }
    if args.device_augment:
        out["e2e"]["host_draw_ms_per_sample"] = legs[0][1].draw_ms_per_sample
    emit(out)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

"""BASELINE.json configs[4]: the BSRGAN full GAN step with the B200 generator and the reference's critics UNCHANGED.

One iteration restates ``BSRGAN/train_bsrgan.py:412-470`` around objects the reference itself defines:

  * ``d_model``          = the reference ``DiscriminatorUNet(3, 1, 64)``            (BSRGAN/model.py:91-167, through the compat shim)
  * ``content_criterion``= the reference ``ContentLoss`` on torchvision VGG19        (BSRGAN/model.py:501-554).  The ImageNet
                           weights are not cached in this image and there is no network, so ``torchvision.models.vgg19`` is
                           patched to return a SEEDED RANDOM-INIT VGG19 (same FLOPs, says so in the output);
  * ``g_model``          = ``bsrgan_x4`` -- the B200 drop-in (``--generator b200``) or the reference's own torch module
                           (``--generator stock``) for the A/B number;
  * autocast + GradScaler(65536), Adam (lr 8e-5, betas (0.9, 0.999), eps 1e-4), D step BETWEEN the generator's forward and its
    backward, generator backward under the summed (pixel 20 + content 1 + adversarial 0.5) x 65536 upstream gradient.

Needs the reference tree (``$SRGANFD_REFERENCE`` or /root/reference) for the critics.  Under torchrun every rank runs 16 images;
the generator's gradients are averaged by ``sr_gan_fd_b200.dist`` (NCCL), the discriminator is wrapped in stock DDP.

    python tools/gan_step.py --steps 10                      # 1 GPU, prints one JSON line
    torchrun --nproc-per-node 8 tools/gan_step.py --steps 10
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch
import torch.distributed as dist
from torch import nn, optim

PIXEL_W, CONTENT_W, ADV_W = [20.0], [1.0], [0.5]                                   # BSRGAN/bsrgan_config.py:137-143
NODES = ["features.2", "features.7", "features.16", "features.25", "features.34"]  # :130
MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]                            # :131-132
LR, BETAS, EPS = 8e-5, (0.9, 0.999), 1e-4                                           # :147-150


def patch_vgg19(seed=1234):
    """torchvision.models.vgg19(weights=IMAGENET1K_V1) would download: return a seeded random-init VGG19 instead."""
    import torchvision.models as models
    real = models.vgg19

    def seeded(*a, **k):
        state = torch.random.get_rng_state()
        torch.manual_seed(seed)
        m = real(weights=None)
        torch.random.set_rng_state(state)
        return m

    models.vgg19 = seeded


def build(generator, device, seed=0, content="reference", disc="reference"):
    patch_vgg19()
    from sr_gan_fd_b200.compat import bsrgan_model as model  # reference critics + B200 generator
    if "discriminator_unet" not in model.__dict__ and (disc == "reference" or content == "reference" or generator == "stock"):
        raise SystemExit("the reference tree is needed for the reference critics / generator (set SRGANFD_REFERENCE), "
                         "or run with --disc b200|torch --content b200|torch")
    torch.manual_seed(seed)
    if disc == "reference":
        d_model = model.discriminator_unet(in_channels=3, out_channels=1, channels=64).to(device)
    else:  # SURVEY 8f rank 2: the drop-in class -- natively (b200) or through its stock torch ops (torch = the reference's op sequence)
        from sr_gan_fd_b200.discriminator import discriminator_unet
        d_model = discriminator_unet(in_channels=3, out_channels=1, channels=64).to(device)
        d_model.use_native = disc == "b200"
    torch.manual_seed(seed)
    if generator == "b200":
        g_model = model.bsrgan_x4(in_channels=3, out_channels=3, channels=64, growth_channels=32, num_rrdb=23)
    else:
        from sr_gan_fd_b200.compat._passthrough import load_reference_model
        g_model = load_reference_model("BSRGAN").bsrgan_x4(in_channels=3, out_channels=3, channels=64, growth_channels=32, num_rrdb=23)
    g_model = g_model.to(device)
    if content in ("b200", "torch"):  # SURVEY 8f rank 3: the same loss on the tcgen05 chain kernel (sr_gan_fd_b200.vgg)
        from sr_gan_fd_b200.vgg import ContentLossMulti
        native = content == "b200"
        content = ContentLossMulti(NODES, MEAN, STD).to(device)
        content.use_native = native
    else:
        content = model.ContentLoss(NODES, MEAN, STD).to(device)
    return d_model, g_model, content


class GanStep:
    def __init__(self, d_model, g_model, content, device, world=1, optimizer="stock", ema=False):
        self.d, self.g, self.content, self.dev = d_model, g_model, content, device
        self.d_core = d_model.module if hasattr(d_model, "module") else d_model
        self.pixel = nn.L1Loss().to(device)
        self.adv = nn.BCEWithLogitsLoss().to(device)
        # EMA copy of the generator as the script keeps it (BSRGAN/train_bsrgan.py:289-291, updated after every generator step, :469)
        self.ema, self.ema_in_optimizer = None, False
        g_core = g_model.module if hasattr(g_model, "module") else g_model
        if ema:
            from torch.optim.swa_utils import AveragedModel
            decay = 0.999  # bsrgan_config.model_ema_decay
            self.ema = AveragedModel(g_core, avg_fn=lambda e, p, n: (1 - decay) * e + decay * p)
        if optimizer == "fused":  # SURVEY 8f rank 1: GradScaler unscale + Adam (+ EMA) as ONE launch per model
            from sr_gan_fd_b200.optim import FusedAdamEMA
            self.d_opt = FusedAdamEMA(self.d_core.parameters(), LR, BETAS, EPS, 0.0)
            self.g_opt = FusedAdamEMA(g_core.parameters(), LR, BETAS, EPS, 0.0, ema_model=self.ema, ema_decay=0.999)
            self.ema_in_optimizer = ema
        else:
            self.d_opt = optim.Adam(self.d_core.parameters(), LR, BETAS, EPS, 0.0)
            self.g_opt = optim.Adam(self.g.parameters(), LR, BETAS, EPS, 0.0)
        self.scaler = torch.amp.GradScaler("cuda")
        self.pw = torch.Tensor(PIXEL_W).to(device)
        self.cw = torch.Tensor(CONTENT_W).to(device)
        self.aw = torch.Tensor(ADV_W).to(device)
        self.sr_grad = None

    def __call__(self, lr, gt, step_d=True, step_g=True, keep_sr_grad=False):
        d_model, g_model, scaler = self.d, self.g, self.scaler
        b, _, h, w = gt.shape
        real_label = torch.full([b, 1, h, w], 1.0, dtype=gt.dtype, device=self.dev)
        fake_label = torch.full([b, 1, h, w], 0.0, dtype=gt.dtype, device=self.dev)
        for p in self.d_core.parameters():
            p.requires_grad = True
        d_model.zero_grad(set_to_none=True)
        with torch.autocast("cuda"):
            gt_output = d_model(gt)
            d_loss_hr = self.adv(gt_output, real_label)
        scaler.scale(d_loss_hr).backward(retain_graph=True)
        with torch.autocast("cuda"):
            sr = g_model(lr)                       # generator forward ONCE; its activations wait for the backward below
            sr_output = d_model(sr.detach().clone())
            d_loss_sr = self.adv(sr_output, fake_label)
        scaler.scale(d_loss_sr).backward()
        if step_d:
            scaler.step(self.d_opt)                # the discriminator changes BETWEEN the generator's forward and backward
            scaler.update()
        for p in self.d_core.parameters():
            p.requires_grad = False
        g_model.zero_grad(set_to_none=True)
        if keep_sr_grad:
            sr.register_hook(lambda gr: setattr(self, "sr_grad", gr.detach().clone()))
        with torch.autocast("cuda"):
            pixel_loss = self.pixel(sr, gt)
            content_loss = self.content(sr, gt)
            adversarial_loss = self.adv(self.d_core(sr), real_label)
            pixel_loss = torch.sum(torch.mul(self.pw, pixel_loss))
            content_loss = torch.sum(torch.mul(self.cw, content_loss))
            adversarial_loss = torch.sum(torch.mul(self.aw, adversarial_loss))
            g_loss = pixel_loss + content_loss + adversarial_loss
        scaler.scale(g_loss).backward()
        if step_g:
            scaler.step(self.g_opt)
            scaler.update()
            if self.ema is not None and not self.ema_in_optimizer:
                self.ema.update_parameters(self.g.module if hasattr(self.g, "module") else self.g)
        return sr, g_loss.detach(), (d_loss_hr + d_loss_sr).detach()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--generator", default="b200", choices=["b200", "stock"])
    ap.add_argument("--content", default="reference", choices=["reference", "b200", "torch"],
                    help="VGG19 content loss: the reference's torch module, sr_gan_fd_b200.vgg natively, or the drop-in's stock torch path")
    ap.add_argument("--disc", default="reference", choices=["reference", "b200", "torch"],
                    help="U-Net discriminator: the reference's torch module, sr_gan_fd_b200.discriminator natively, or the drop-in's stock torch path")
    ap.add_argument("--optim", default="stock", choices=["stock", "fused"], help="torch.optim.Adam as the script, or sr_gan_fd_b200.optim.FusedAdamEMA")
    ap.add_argument("--ema", action="store_true", help="keep the generator's EMA copy as the script does (AveragedModel.update_parameters, or inside the fused step)")
    ap.add_argument("--profile", default="", help="write a per-kernel GPU-time table of ONE extra step (torch.profiler) to this file")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--lr-size", type=int, default=64)
    ap.add_argument("--deterministic", action="store_true",
                    help="torch.use_deterministic_algorithms(True): bit-reproducible steps (needs CUBLAS_WORKSPACE_CONFIG=:4096:8)")
    args = ap.parse_args()
    if args.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # torch's own cuBLAS calls (spectral norm) demand it
        torch.use_deterministic_algorithms(True)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    d_model, g_model, content = build(args.generator, dev, content=args.content, disc=args.disc)
    d_model.train(); g_model.train()
    if world > 1:
        d_model = nn.parallel.DistributedDataParallel(d_model, device_ids=[local], broadcast_buffers=True)
        if args.generator == "b200":
            from sr_gan_fd_b200 import dist as b200dist
            b200dist.make_data_parallel(g_model)
        else:
            g_model = nn.parallel.DistributedDataParallel(g_model, device_ids=[local])
    step = GanStep(d_model, g_model, content, dev, world, optimizer=args.optim, ema=args.ema)
    torch.manual_seed(100 + rank)
    lr = torch.rand(args.batch, 3, args.lr_size, args.lr_size, device=dev)
    gt = torch.rand(args.batch, 3, 4 * args.lr_size, 4 * args.lr_size, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(lr, gt)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        _, g_loss, d_loss = step(lr, gt)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if rank == 0:
        print(json.dumps({
            "metric": "BSRGAN full GAN step imgs/s (BASELINE configs[4]: generator fwd+bwd + reference U-Net discriminator x3 + VGG19 content loss)",
            "generator": args.generator, "content_loss": args.content, "discriminator": args.disc, "optimizer": args.optim, "ema": bool(args.ema), "value": world * args.batch / (ms * 1e-3), "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "deterministic": bool(args.deterministic), "higher_is_better": True, "scaling": "weak", "data": "synthetic",
            "config": {"batch_per_gpu": args.batch, "lr": args.lr_size, "scale": 4, "num_rrdb": 23, "critics": "reference DiscriminatorUNet(3,1,64) "
                       "+ ContentLoss on a SEEDED RANDOM-INIT VGG19 (ImageNet weights unavailable offline), autocast fp16 + GradScaler",
                       "discriminator_parallelism": "stock DDP" if world > 1 else "single", "g_loss": float(g_loss), "d_loss": float(d_loss)}}), flush=True)
    if args.profile and rank == 0:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            step(lr, gt)
            torch.cuda.synchronize()
        rows = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                r = rows.setdefault(ev.name[:70], [0.0, 0])
                r[0] += ev.device_time
                r[1] += 1
        total = sum(r[0] for r in rows.values())
        with open(args.profile, "w") as fh:
            fh.write(f"GPU kernel time of one step: {total / 1e3:.2f} ms in {sum(r[1] for r in rows.values())} launches (step wall {ms:.2f} ms)\n")
            for name, (t, c) in sorted(rows.items(), key=lambda kv: -kv[1][0])[:45]:
                fh.write(f"{t / 1e3:9.3f} ms {c:5d} x  {name}\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

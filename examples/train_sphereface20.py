#!/usr/bin/env python
"""End-to-end glue (SURVEY.md section 8f rank 4; BASELINE config 2): a stock torch/cuDNN
restatement of the reference's SphereFaceNet-20 backbone (nets/sphere.py:23-76) feeding the
B200 A-softmax head, driven like the reference's train loop (train.py:223-250).

    python examples/train_sphereface20.py --steps 20 --batch 512 --classes 10572
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 \
        examples/train_sphereface20.py --batch 512        # DDP backbone + class-sharded head
    python examples/train_sphereface20.py --margin arcface --scale 64 --margin-value 0.5
    python examples/train_sphereface20.py --loss focal --focal-gamma 1 --focal-alpha 2

Only the head is this repository's product; the backbone is ordinary PyTorch (the survey
marks backbones out of scope) and exists to show where the head plugs in:
  features = backbone(images)                                   nets/sphere.py:82
  loss, _, dX, _ = asoftmax_head(features, labels, C, m, lambda, weights=W, optimizer=opt)
  features.backward(dX)                                         data_parallel.py:32-38
Synthetic 112x96 faces; prints loss and images/s like train.py:231-239.
"""
import argparse
import os
import sys
import time

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tf_face_toolbox_b200 import AdditiveMargin, FocalLoss, FusedOptimizer, LambdaState, asoftmax_head  # noqa: E402


class ResBlock(nn.Module):
    """Two 3x3 convs with PReLU and an identity shortcut (nets/sphere.py:38-45)."""

    def __init__(self, ch):
        super().__init__()
        self.c1, self.a1 = nn.Conv2d(ch, ch, 3, padding=1), nn.PReLU(ch)
        self.c2, self.a2 = nn.Conv2d(ch, ch, 3, padding=1), nn.PReLU(ch)

    def forward(self, x):
        return x + self.a2(self.c2(self.a1(self.c1(x))))


class SphereFaceNet20(nn.Module):
    """Stages [64,128,256,512], each a stride-2 3x3 conv + {1,2,4,1} residual blocks, then
    flatten -> FC 512 (nets/sphere.py:47-76).  112x96 input -> 7x6x512 -> 512-d embedding."""

    def __init__(self, emb=512):
        super().__init__()
        layers, cin = [], 3
        for ch, nblk in zip((64, 128, 256, 512), (1, 2, 4, 1)):
            layers += [nn.Conv2d(cin, ch, 3, stride=2, padding=1), nn.PReLU(ch)]
            layers += [ResBlock(ch) for _ in range(nblk)]
            cin = ch
        self.body = nn.Sequential(*layers)
        self.fc = nn.Linear(512 * 7 * 6, emb)

    def forward(self, x):
        return self.fc(torch.flatten(self.body(x), 1))


def head_step(net, images, labels, head_call, opt_backbone, world=1, clip=5.0, autocast=True):
    """One training step of the reference-shaped loop (data_parallel.py:203-256) around the head.

    `head_call(features, labels) -> (loss, dX)` runs the A-softmax head (and its optimizer);
    dX is d(global-batch mean loss)/d(features of THIS rank's rows).  With a data-parallel
    backbone (DDP averages gradients over ranks) the backbone gradient of the global mean is
    the SUM of the ranks' contributions, hence the `* world` -- the mirror image of the
    reference's `grad *= 1/num_gpus` followed by `nccl.all_sum` (data_parallel.py:37, 179)."""
    if autocast and images.is_cuda:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            feats = net(images)
    else:
        feats = net(images)
    feats32 = feats.float()
    loss, dX = head_call(feats32.detach(), labels)
    opt_backbone.zero_grad(set_to_none=True)
    feats32.backward(dX * world if world > 1 else dX)
    if clip:
        torch.nn.utils.clip_grad_norm_(net.parameters(), clip)    # un-normalised synthetic net
    opt_backbone.step()
    return loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=512, help="GLOBAL batch (train.py: batch_size)")
    ap.add_argument("--classes", type=int, default=10572)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--mode", default="bf16")
    ap.add_argument("--transport", default="nvlink", help="multi-GPU exchanges: nvlink | nccl")
    ap.add_argument("--margin", default="asoftmax", choices=["asoftmax", "arcface", "cosface"],
                    help="A-softmax (m = 4, annealed lambda), or an additive margin on normalised embeddings")
    ap.add_argument("--scale", type=float, default=64.0, help="s of the additive margins")
    ap.add_argument("--margin-value", type=float, default=None,
                    help="m2 of ArcFace (default 0.5) or m3 of CosFace (default 0.35)")
    ap.add_argument("--loss", default="ce", choices=["ce", "focal"],
                    help="softmax cross-entropy, or the reference's focal loss gamma (1 - p)^alpha CE")
    ap.add_argument("--focal-gamma", type=float, default=1.0, help="gamma of the focal loss: the multiplier")
    ap.add_argument("--focal-alpha", type=float, default=2.0, help="alpha of the focal loss: the exponent")
    args = ap.parse_args()
    loss_kind = FocalLoss(args.focal_gamma, args.focal_alpha) if args.loss == "focal" else None
    if args.margin == "arcface":
        margin = AdditiveMargin.arcface(args.scale, 0.5 if args.margin_value is None else args.margin_value)
    elif args.margin == "cosface":
        margin = AdditiveMargin.cosface(args.scale, 0.35 if args.margin_value is None else args.margin_value)
    else:
        margin = None
    # under torchrun: data-parallel backbone (DDP) + class-parallel head, one rank per GPU
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    net = SphereFaceNet20().to(dev).to(memory_format=torch.channels_last)
    if world > 1:
        net = nn.parallel.DistributedDataParallel(net, device_ids=[local])
    opt_backbone = torch.optim.SGD(net.parameters(), lr=args.lr, momentum=0.9, weight_decay=5e-4)
    opt_head = FusedOptimizer("Momentum", lr=args.lr, weight_decay=5e-4)
    lam = LambdaState()                                               # global_step clock
    b_local = args.batch // world
    if world > 1:
        from tf_face_toolbox_b200 import ShardedASoftmaxHead
        head = ShardedASoftmaxHead(512, args.classes, m=4, mode=args.mode, device=dev, lambda_state=lam,
                                   transport=args.transport, batch_global=args.batch,   # N(0, 0.001) shards
                                   margin=margin, loss=loss_kind)

        def head_call(feats, labels):
            loss, dX, _ = head.step(feats, labels, optimizer=opt_head)                  # lambda from the clock
            return loss, dX
    else:
        W = (torch.randn(512, args.classes, device=dev) * 0.001)      # nets/sphere.py:87

        def head_call(feats, labels):
            loss, _, dX, _ = asoftmax_head(feats, labels, args.classes, 4, lam.step(),
                                           weights=W, mode=args.mode, optimizer=opt_head, margin=margin,
                                           loss=loss_kind)
            return loss, dX
    # a fixed synthetic "dataset" of 4 batches so the loss can actually go down; every rank draws
    # the same global batch and keeps its slice (data_parallel.py:206-207)
    g = torch.Generator(device="cpu").manual_seed(1)
    data = []
    for _ in range(4):
        imgs = torch.randn(args.batch, 3, 112, 96, generator=g)[rank * b_local:(rank + 1) * b_local]
        labs = torch.randint(0, args.classes, (args.batch,), generator=g, dtype=torch.int32)[rank * b_local:(rank + 1) * b_local]
        data.append((imgs.to(dev).contiguous(memory_format=torch.channels_last), labs.to(dev)))
    losses = []
    t0 = None
    for step in range(args.steps):
        if step == 3:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        images, labels = data[step % len(data)]
        loss = head_step(net, images, labels, head_call, opt_backbone, world=world)
        losses.append(loss)
        if rank == 0 and (step % 5 == 0 or step == args.steps - 1):
            extra = f"  lambda {lam.value():.2f}" if margin is None else f"  {args.margin} s={margin.s:g}"
            name = "focal_loss" if loss_kind is not None else "cross_entropy"
            print(f"step {step:4d}  {name} {float(loss):.4f}{extra}", flush=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    first, last = float(torch.stack(losses[:4]).mean()), float(torch.stack(losses[-4:]).mean())
    if rank == 0:
        # train.py:231-239 prints batch_size / duration with the GLOBAL batch
        print(f"{(args.steps - 3) * args.batch / dt:.1f} images/s  ({1e3 * dt / (args.steps - 3):.1f} ms/batch, {world} GPU)")
        print(f"mean loss first 4 steps {first:.4f} -> last 4 steps {last:.4f}")
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return first, last


if __name__ == "__main__":
    main()

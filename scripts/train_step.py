#!/usr/bin/env python
"""BASELINE config 4: the reference's train step on N B200s -- `train.py:755-773` (autocast forward of the two-stream
model, `ComputeLoss` of `utils/loss.py:88-216`, backward, SGD + nesterov `train.py:560`) under data parallelism
(`train.py:654-658`), bf16 autocast, global batch = 32 x N, 640 x 640 synthetic RGB+IR pairs and labels.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           scripts/train_step.py [--batch 32] [--steps 6] [--warmup 2] [--cfg yolov5l_fusion_transformerx3_FLIR_aligned]

What runs where.  The model, the loss and the backward are the UNMODIFIED reference's own PyTorch modules / autograd
(from the reference tree, or its staged copy oracle/_ref on the GPU machine): this repository has no backward kernels
(DESIGN.md section 6), and its forward kernels are eval-only (BatchNorm running statistics folded), so the train-mode
forward is the reference's too.  What this repository contributes to the step is the one exchange of the path: the
gradient all-reduce (`allreduce.GradientAllReduce`, NCCL over NVLink / NVSwitch).  Three variants of the same step are timed,
CUDA events, max over ranks, and rank 0 prints one JSON line each:

  no_comm   forward + backward + optimizer step, no gradient exchange at all (the compute floor of the step)
  ddp       the reference's way: torch DistributedDataParallel (fp32 buckets of 25 MiB, reduced from inside backward)
  gar       GradientAllReduce.attach(): bucketed all-reduce launched from post-accumulate-grad hooks on a side stream,
            fp32 wire format (--wire bf16 halves the bytes), finish() before the optimizer step
plus the exchange alone (`allreduce_only`: reduce() on ready gradients).  exposed = step - no_comm;
overlap fraction = 1 - exposed / allreduce_only.
"""
import argparse
import importlib
import json
import os
import sys

import torch
import torch.distributed as dist
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# data/hyp.scratch.yaml:6-22 of the reference (the default --hyp of train.py)
HYP = {"lr0": 0.01, "lrf": 0.2, "momentum": 0.937, "weight_decay": 0.0005, "box": 0.05, "cls": 0.5, "cls_pw": 1.0,
       "obj": 1.0, "obj_pw": 1.0, "iou_t": 0.20, "anchor_t": 4.0, "fl_gamma": 0.0, "label_smoothing": 0.0}


def build(cfg_name, dev, world, batch, img):
    from oracle import ref_shim
    yt = ref_shim.import_reference()
    model = yt.Model(ref_shim.reference_yaml(cfg_name), ch=3).to(dev)
    det = model.model[-1]
    nl, nc = det.nl, det.nc
    hyp = dict(HYP)
    total = batch * world
    hyp["weight_decay"] *= total * max(round(64 / total), 1) / 64          # train.py:543-545
    hyp["box"] *= 3.0 / nl                                                  # train.py:661-664
    hyp["cls"] *= nc / 80.0 * 3.0 / nl
    hyp["obj"] *= (img / 640) ** 2 * 3.0 / nl
    model.nc, model.hyp, model.gr = nc, hyp, 1.0                            # train.py:665-668
    pg0, pg1, pg2 = [], [], []                                              # train.py:548-556
    for _, v in model.named_modules():
        if hasattr(v, "bias") and isinstance(v.bias, nn.Parameter):
            pg2.append(v.bias)
        if isinstance(v, nn.BatchNorm2d):
            pg0.append(v.weight)
        elif hasattr(v, "weight") and isinstance(v.weight, nn.Parameter):
            pg1.append(v.weight)
    opt = torch.optim.SGD(pg0, lr=hyp["lr0"], momentum=hyp["momentum"], nesterov=True)     # train.py:560
    opt.add_param_group({"params": pg1, "weight_decay": hyp["weight_decay"]})
    opt.add_param_group({"params": pg2})
    from utils.loss import ComputeLoss                                      # the reference's loss (utils/loss.py:88)

    class ComputeLossT2(ComputeLoss):
        """The reference's ComputeLoss with `build_targets` (utils/loss.py:163-216) restated: the original clamps LONG grid
        indices with FLOAT tensor bounds (`gj.clamp_(0, gain[3] - 1)`, :211), which PyTorch >= 1.10 rejects ("result type
        Float can't be cast to ... long"); here the bounds are Python ints.  Same matching rule otherwise: a label is
        assigned to anchor a of level i when max(wh / anchor, anchor / wh) < anchor_t, to its own cell and to the up-to-two
        neighbour cells whose centre is nearest (offsets of 0.5)."""

        def build_targets(self, p, targets):
            dev, na, nt = targets.device, self.na, targets.shape[0]
            tcls, tbox, indices, anch = [], [], [], []
            ai = torch.arange(na, device=dev, dtype=torch.float32).view(na, 1).expand(na, nt)
            tg = torch.cat((targets.unsqueeze(0).expand(na, nt, 6), ai.unsqueeze(2)), 2)      # [na, nt, 7]: + anchor index
            off = 0.5 * torch.tensor([[0, 0], [1, 0], [0, 1], [-1, 0], [0, -1]], device=dev, dtype=torch.float32)
            for i in range(self.nl):
                anchors = self.anchors[i]
                ny, nx = int(p[i].shape[2]), int(p[i].shape[3])
                scale = torch.tensor([1, 1, nx, ny, nx, ny, 1], device=dev, dtype=torch.float32)
                t = tg * scale
                if nt:
                    r = t[:, :, 4:6] / anchors[:, None]
                    t = t[torch.max(r, 1.0 / r).max(2)[0] < self.hyp["anchor_t"]]
                    gxy = t[:, 2:4]
                    gxi = scale[[2, 3]] - gxy
                    j, k = ((gxy % 1.0 < 0.5) & (gxy > 1.0)).T
                    l, m = ((gxi % 1.0 < 0.5) & (gxi > 1.0)).T
                    sel = torch.stack((torch.ones_like(j), j, k, l, m))
                    t = t.repeat((5, 1, 1))[sel]
                    offsets = (torch.zeros_like(gxy)[None] + off[:, None])[sel]
                else:
                    t, offsets = tg[0], 0
                b, c = t[:, :2].long().T
                gxy, gwh = t[:, 2:4], t[:, 4:6]
                gij = (gxy - offsets).long()
                gi, gj = gij.T
                a = t[:, 6].long()
                indices.append((b, a, gj.clamp(0, ny - 1), gi.clamp(0, nx - 1)))
                tbox.append(torch.cat((gxy - gij, gwh), 1))
                anch.append(anchors[a])
                tcls.append(c)
            return tcls, tbox, indices, anch

    return model, opt, ComputeLossT2(model)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default="yolov5l_fusion_transformerx3_FLIR_aligned")
    ap.add_argument("--batch", type=int, default=32, help="pairs per GPU")
    ap.add_argument("--img", type=int, default=640)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--wire", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--modes", default="no_comm,ddp,gar")
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ar = importlib.import_module("multispectral-object-detection_b200.allreduce")
    torch.manual_seed(0)
    model, opt, compute_loss = build(args.cfg, dev, world, args.batch, args.img)
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    n_params = sum(p.numel() for p in params)

    g = torch.Generator().manual_seed(1 + rank)
    B, H = args.batch, args.img
    imgs = torch.randint(0, 256, (B, 6, H, H), dtype=torch.uint8, generator=g).to(dev)
    nt = 8 * B                                                               # 8 labelled boxes per pair
    targets = torch.cat([torch.randint(0, B, (nt, 1), generator=g).float(),
                         torch.randint(0, model.nc, (nt, 1), generator=g).float(),
                         torch.rand(nt, 2, generator=g) * 0.8 + 0.1, torch.rand(nt, 2, generator=g) * 0.3 + 0.02], 1).to(dev)

    ddp = None
    red = ar.GradientAllReduce(params, dtype=torch.bfloat16 if args.wire == "bf16" else None)

    def fwd_bwd(net):
        x = imgs.float() / 255.0                                             # train.py:715
        with torch.autocast("cuda", dtype=torch.bfloat16):
            pred = net(x[:, :3], x[:, 3:])                                   # train.py:757
            loss, _ = compute_loss(pred, targets)                            # train.py:758
            if world > 1:
                loss = loss * world                                          # train.py:759-760
        loss.backward()
        return loss.detach()

    def step(mode):
        if mode == "ddp":
            loss = fwd_bwd(ddp)
        elif mode == "gar":
            red.attach()
            loss = fwd_bwd(model)
            red.finish()
        else:
            red.detach()
            loss = fwd_bwd(model)
        opt.step()                                                           # train.py:766
        opt.zero_grad(set_to_none=False)
        return loss

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    out = {"what": "BASELINE config 4 train step (reference modules + autograd, bf16 autocast, SGD nesterov)", "cfg": args.cfg,
           "n_gpus": world, "batch_per_gpu": B, "global_batch": B * world, "img": H, "params": n_params,
           "grad_bytes_fp32": n_params * 4, "wire": args.wire, "steps": args.steps}
    modes = [m for m in args.modes.split(",") if m]
    if "no_comm" in modes:
        out["no_comm_ms"] = timed(lambda: step("no_comm"), args.steps, args.warmup)
    red.detach()
    # the exchange alone, on ready gradients
    for p in params:
        if p.grad is None:
            p.grad = torch.zeros_like(p)
    out["allreduce_only_ms"] = timed(red.reduce, 10, 3) if world > 1 else 0.0
    if world > 1:
        out["allreduce_busbw_gbs"] = 2.0 * (world - 1) / world * red.wire_bytes() / (out["allreduce_only_ms"] / 1e3) / 1e9
    if "gar" in modes:
        out["gar_ms"] = timed(lambda: step("gar"), args.steps, args.warmup)
        red.detach()
    if "ddp" in modes and world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP
        ddp = DDP(model, device_ids=[local], output_device=local)           # train.py:655-658
        out["ddp_ms"] = timed(lambda: step("ddp"), args.steps, args.warmup)
    if rank == 0:
        base = out.get("no_comm_ms")
        for k in ("gar", "ddp"):
            if base and k + "_ms" in out and out.get("allreduce_only_ms"):
                exposed = max(out[k + "_ms"] - base, 0.0)
                out[k + "_exposed_ms"] = exposed
                out[k + "_overlap_frac"] = 1.0 - min(exposed / out["allreduce_only_ms"], 1.0)
                out[k + "_pairs_per_s"] = B * world / (out[k + "_ms"] / 1e3)
        if base:
            out["no_comm_pairs_per_s"] = B * world / (base / 1e3)
        out["mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

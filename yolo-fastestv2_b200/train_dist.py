#!/usr/bin/env python
"""Multi-GPU launcher for the reference's training loop (SURVEY 8f.1; the reference's train.py is single-device).

    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 yolo-fastestv2_b200/train_dist.py --data data/coco.data

One process per GPU.  Everything that is not the hot path keeps the reference's semantics, line for line where it can:
  * config, datasets, collate_fn, evaluation: the reference's own modules (utils.utils / utils.datasets, resolved from the
    reference checkout on PYTHONPATH, exactly as train.py resolves them), so the `.data` file is the configuration surface;
  * loaders as train.py:34-58, the train loader behind a DistributedSampler (each rank draws batch_size / subdivisions
    images per iteration, as the single-device loop does, so the global batch is world_size times the reference's);
  * the loop of train.py:95-131: `imgs.float() / 255`, forward, compute_loss, backward, the 5-epoch quartic warm-up of
    :113-119, `subdivisions` gradient accumulation (:122-124), MultiStepLR per epoch (:147);
  * rank 0 alone evaluates and saves every 10th epoch (train.py:134-144).
What changes is the hot path: model.detector.Detector / utils.loss.compute_loss are the CUDA mirrors, all gradients live in
one flat 243 095-float bucket and every optimizer step issues exactly ONE all-reduce over NCCL (mean over ranks), then the
reference's SGD.  BatchNorm statistics stay per rank (the reference has no SyncBN).

`--synthetic N` replaces the dataset by N seeded synthetic images with SURVEY 8(d) config[2] box statistics (no dataset and
no reference checkout needed: used by the GPU tests and the 8-GPU measurement)."""
import argparse
import math
import os
import sys
import time

_PKG = os.path.dirname(os.path.abspath(__file__))
if _PKG not in sys.path:
    sys.path.insert(0, _PKG)

import torch                                    # noqa: E402
import torch.distributed as dist                # noqa: E402
from torch.utils.data import DataLoader         # noqa: E402
from torch.utils.data.distributed import DistributedSampler   # noqa: E402

import train_ddp                                # noqa: E402


class SyntheticDetection(torch.utils.data.Dataset):
    """uint8 CHW images + rows (0, cls, cx, cy, w, h), the shapes utils.datasets.TensorDataset yields (datasets.py:100-126)."""

    def __init__(self, n, width, height, classes, seed=2):
        self.n, self.w, self.h, self.classes, self.seed = n, width, height, classes, seed

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(self.seed * 1000003 + i)
        img = torch.randint(0, 256, (3, self.h, self.w), generator=g, dtype=torch.uint8)
        k = int(torch.randint(1, 14, (1,), generator=g))
        t = torch.zeros((k, 6))
        t[:, 1] = torch.randint(0, self.classes, (k,), generator=g).float()
        t[:, 2:4] = torch.rand((k, 2), generator=g)
        t[:, 4:6] = 0.02 + 0.5 * torch.rand((k, 2), generator=g)
        return img, t


class SyntheticRawDetection(SyntheticDetection):
    """Decoded-image form of SyntheticDetection for --device-resize: uint8 HWC images of seeded sizes (as cv2.imread returns
    them, before any resize) with the same kind of label rows."""

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(self.seed * 1000003 + i)
        h, w = int(torch.randint(96, 641, (1,), generator=g)), int(torch.randint(96, 641, (1,), generator=g))
        _, t = super().__getitem__(i)
        return torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8), t


def collate_fn(batch):
    """utils/datasets.py:127-135: image index into column 0, targets concatenated."""
    imgs, targets = list(zip(*batch))
    for i, boxes in enumerate(targets):
        boxes[:, 0] = i
    return torch.stack(imgs), torch.cat(targets, 0)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--data", type=str, default="", help="training profile *.data (as train.py)")
    ap.add_argument("--synthetic", type=int, default=0, help="use N synthetic images instead of cfg['train']")
    ap.add_argument("--epochs", type=int, default=None, help="override cfg['epochs']")
    ap.add_argument("--max-iters", type=int, default=None, help="stop after this many iterations (smoke runs)")
    ap.add_argument("--save-dir", type=str, default="weights")
    ap.add_argument("--device-aug", action="store_true", help="run contrast_and_brightness (utils/datasets.py:10-16) on the uint8 batch "
                                                              "on the GPU (csrc/k_aug.cu) instead of per image in the data-loader workers")
    ap.add_argument("--device-resize", action="store_true", help="data-loader workers only decode; the cv2.resize of "
                                                                 "utils/datasets.py:106-111 runs on the GPU (csrc/k_resize.cu), followed by "
                                                                 "contrast_and_brightness for the training batches")
    opt = ap.parse_args(argv)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("train_dist.py: the hot path runs on CUDA only (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    import utils.utils
    import utils.loss
    import model.detector
    cfg = utils.utils.load_datafile(opt.data)
    if rank == 0:
        print("training configuration:", cfg, "| world size", world)

    batch_size = int(cfg["batch_size"] / cfg["subdivisions"])                     # per rank, as train.py:37
    nw = min([os.cpu_count(), batch_size if batch_size > 1 else 0, 8])
    if opt.device_resize:
        import utils.device_aug
        cf = utils.device_aug.collate_packed
        if opt.synthetic:
            train_dataset, val_dataset = SyntheticRawDetection(opt.synthetic, cfg["width"], cfg["height"], cfg["classes"]), None
        else:
            train_dataset = utils.device_aug.RawImageDataset(cfg["train"], cfg["width"], cfg["height"])
            val_dataset = utils.device_aug.RawImageDataset(cfg["val"], cfg["width"], cfg["height"])
    elif opt.synthetic:
        train_dataset = SyntheticDetection(opt.synthetic, cfg["width"], cfg["height"], cfg["classes"])
        val_dataset, cf = None, collate_fn
    else:
        import utils.datasets                                                     # the reference's (not on the hot path)
        train_dataset = utils.datasets.TensorDataset(cfg["train"], cfg["width"], cfg["height"], imgaug=not opt.device_aug)
        val_dataset = utils.datasets.TensorDataset(cfg["val"], cfg["width"], cfg["height"], imgaug=False)
        cf = utils.datasets.collate_fn
    sampler = DistributedSampler(train_dataset, num_replicas=world, rank=rank, shuffle=True, drop_last=True)
    train_dataloader = DataLoader(train_dataset, batch_size=batch_size, sampler=sampler, collate_fn=cf, num_workers=nw,
                                  pin_memory=True, drop_last=True, persistent_workers=nw > 0)
    val_dataloader = None
    if val_dataset is not None and rank == 0:
        val_dataloader = DataLoader(val_dataset, batch_size=batch_size, shuffle=False, collate_fn=cf, num_workers=nw,
                                    pin_memory=True, drop_last=False, persistent_workers=nw > 0)
    if opt.device_resize:
        # the reference augments every training image (train.py: TensorDataset(..., imgaug=True)); synthetic data only with --device-aug
        train_dataloader = utils.device_aug.DeviceResizeLoader(train_dataloader, cfg["width"], cfg["height"], device,
                                                               imgaug=opt.device_aug or not opt.synthetic)
        if val_dataloader is not None:
            val_dataloader = utils.device_aug.DeviceResizeLoader(val_dataloader, cfg["width"], cfg["height"], device)

    load_param = bool(cfg["pre_weights"]) and os.path.exists(cfg["pre_weights"])
    torch.manual_seed(0)                                                          # identical initial weights on every rank
    # load_param=False makes the constructor read ./model/backbone/backbone.pth from the reference checkout (shufflenetv2.py);
    # synthetic runs outside a checkout keep the seeded default initialisation instead
    ctor_load = load_param or (bool(opt.synthetic) and not os.path.exists("./model/backbone/backbone.pth"))
    net = model.detector.Detector(cfg["classes"], cfg["anchor_num"], ctor_load).to(device)
    if load_param:
        net.load_state_dict(torch.load(cfg["pre_weights"], map_location=device), strict=False)
    if world > 1:                                                                 # belt and braces: rank 0's weights everywhere
        for t in list(net.parameters()) + list(net.buffers()):
            dist.broadcast(t.data, src=0)

    bucket = train_ddp.FlatGradBucket(net.parameters())
    optimizer = train_ddp.make_optimizer(net, cfg["learning_rate"])               # train.py:81-85
    scheduler = torch.optim.lr_scheduler.MultiStepLR(optimizer, milestones=[int(s) for s in cfg["steps"]], gamma=0.1)

    epochs = opt.epochs if opt.epochs is not None else cfg["epochs"]
    batch_num, t0, seen = 0, time.time(), 0
    bucket.zero()
    for epoch in range(epochs):
        net.train()
        sampler.set_epoch(epoch)
        for imgs, targets in train_dataloader:
            imgs = imgs.to(device, non_blocking=True)
            if opt.device_aug and not opt.device_resize and imgs.dtype == torch.uint8:   # (DeviceResizeLoader augments itself)
                import utils.device_aug
                imgs = utils.device_aug.img_aug_batch(imgs, out=imgs)                 # datasets.py:63-68 on the device, in place
            imgs = imgs.float() / 255.0                                           # train.py:101
            targets = targets.to(device, non_blocking=True)
            preds = net(imgs)
            iou_loss, obj_loss, cls_loss, total_loss = utils.loss.compute_loss(preds, targets, cfg, device)
            total_loss.backward()                                                 # accumulates into the flat bucket
            for g in optimizer.param_groups:                                      # warm-up, train.py:113-119
                warmup_num = 5 * len(train_dataloader)
                if batch_num <= warmup_num:
                    g["lr"] = cfg["learning_rate"] * math.pow(batch_num / warmup_num, 4)
                lr = g["lr"]
            if batch_num % cfg["subdivisions"] == 0:                              # train.py:122-124
                bucket.allreduce_mean()                                           # the single collective of the step
                optimizer.step()
                bucket.zero()                                                     # (= optimizer.zero_grad() with the views kept)
            seen += imgs.shape[0] * world
            if rank == 0 and batch_num % 10 == 0:
                print("Epoch:%d it:%d LR:%f CIou:%f Obj:%f Cls:%f Total:%f  %.0f img/s" % (
                    epoch, batch_num, lr, iou_loss, obj_loss, cls_loss, total_loss, seen / max(time.time() - t0, 1e-9)), flush=True)
            batch_num += 1
            if opt.max_iters is not None and batch_num >= opt.max_iters:
                break
        if epoch % 10 == 0 and epoch > 0 and rank == 0 and val_dataloader is not None:      # train.py:134-144
            net.eval()
            _, _, AP, _ = utils.utils.evaluation(val_dataloader, cfg, net, device)
            precision, recall, _, f1 = utils.utils.evaluation(val_dataloader, cfg, net, device, 0.3)
            print("Precision:%f Recall:%f AP:%f F1:%f" % (precision, recall, AP, f1))
            os.makedirs(opt.save_dir, exist_ok=True)
            torch.save(net.state_dict(), os.path.join(opt.save_dir, "%s-%d-epoch-%fap-model.pth" % (cfg["model_name"], epoch, AP)))
        if world > 1:
            dist.barrier()                                                        # the other ranks wait for rank 0's evaluation
        scheduler.step()
        if opt.max_iters is not None and batch_num >= opt.max_iters:
            break
    if world > 1:
        dist.destroy_process_group()
    return net


if __name__ == "__main__":
    main()

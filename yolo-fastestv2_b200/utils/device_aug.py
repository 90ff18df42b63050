"""Batch-level, on-device form of the reference's img_aug (utils/datasets.py:63-68 -> contrast_and_brightness, :10-16).

The reference augments each uint8 HWC image on the host inside TensorDataset.__getitem__; with the input pipeline moved to the
GPU (uint8 batch copied first, `/255` fused into the stem) the same byte arithmetic runs on the whole uint8 batch in one
kernel of libyfv2.so (csrc/k_aug.cu), bit-identical to cv2.addWeighted.  (alpha, beta) are drawn per image from the same
random.uniform(0.25, 1.75) calls, in the same order as the reference would draw them image by image."""
import random

import torch

import yfv2_engine


def img_aug_batch(imgs_u8, rng=random, out=None):
    """imgs_u8: CUDA uint8 [N, ...] (any per-image layout).  Returns the augmented batch (new tensor unless `out` is given)."""
    n = imgs_u8.shape[0]
    ab = [(rng.uniform(0.25, 1.75), rng.uniform(0.25, 1.75)) for _ in range(n)]      # alpha first, then beta (datasets.py:11-12)
    alpha = torch.tensor([a for a, _ in ab], dtype=torch.float32)
    beta = torch.tensor([b for _, b in ab], dtype=torch.float32)
    return yfv2_engine.contrast_and_brightness(imgs_u8, alpha, beta, out=out)


# ---- decoded images at original size -> one packed host buffer -> resized on the device ---------------------------------------
# The reference resizes every decoded image on the host (utils/datasets.py:106-111: cv2.imread -> cv2.resize(INTER_LINEAR) ->
# img_aug -> transpose).  Here the data-loader workers only decode; the collate packs the ragged batch into ONE uint8 buffer (the
# DataLoader pins it, the loop makes one host-to-device copy) and yfv2_resize_u8 (csrc/k_resize.cu, bit-identical to cv2.resize)
# produces the [N,3,H,W] uint8 batch on the GPU.  Decoding stays on the host.
import os  # noqa: E402


def label_path_for(img_path):
    """The label file the reference pairs with an image: the path up to its first '.', plus '.txt' (utils/datasets.py:101)."""
    return img_path.split(".")[0] + ".txt"


def read_darknet_labels(path):
    """A darknet label file (one `class cx cy w h` line per box, normalised) as float32 rows (0, class, cx, cy, w, h), the rows
    TensorDataset yields; a missing file is an error, as in the reference."""
    if not os.path.exists(path):
        raise Exception("%s is not exist" % path)
    rows = []
    with open(path, "r") as f:
        for line in f:
            fields = line.split()
            if not fields:
                continue
            if len(fields) != 5:
                raise ValueError("%s: expected 5 label columns, got %d" % (path, len(fields)))
            rows.append([0.0] + [float(v) for v in fields])
    return torch.tensor(rows, dtype=torch.float32).reshape(-1, 6)


def _raw_image_dataset_class():
    import cv2
    from utils.datasets import TensorDataset          # the reference's (resolved from its checkout, utils/__init__.py)

    class RawImageDataset(TensorDataset):
        """TensorDataset (same list-file checks, same label rows) that returns the decoded BGR image at its original size as a
        uint8 [h, w, 3] tensor: the resize (and the augmentation) run on the device, see DeviceResizeLoader."""

        def __init__(self, path, img_size_width=352, img_size_height=352):
            super().__init__(path, img_size_width, img_size_height, imgaug=False)

        def __getitem__(self, index):
            img_path = self.data_list[index]
            img = cv2.imread(img_path)
            if img is None:
                raise Exception("cannot decode %s" % img_path)
            return torch.from_numpy(img), read_darknet_labels(label_path_for(img_path))

    return RawImageDataset


def __getattr__(name):
    # RawImageDataset subclasses the reference's TensorDataset, so it exists where the reference checkout (and cv2) does
    if name == "RawImageDataset":
        cls = _raw_image_dataset_class()
        globals()[name] = cls
        return cls
    raise AttributeError(name)


def collate_packed(batch):
    """collate_fn for (uint8 [h, w, 3] image, label rows) samples of any sizes: (packed uint8 [sum 3hw] buffer, sizes int64 [N, 2]
    of (h, w), targets [nt, 6] with the image index stamped into column 0 as utils/datasets.py:127-132 does).  Images follow each
    other byte by byte, so most start at unaligned offsets; yfv2_resize_u8 takes that."""
    imgs, labels = zip(*batch)
    sizes = torch.tensor([[im.shape[0], im.shape[1]] for im in imgs], dtype=torch.int64)
    packed = torch.empty(sum(im.numel() for im in imgs), dtype=torch.uint8)
    off = 0
    for im in imgs:
        packed[off:off + im.numel()] = im.reshape(-1)
        off += im.numel()
    for i, lab in enumerate(labels):
        if lab.shape[0] > 0:
            lab[:, 0] = i
    return packed, sizes, torch.cat(labels, 0)


def unpack(packed, sizes):
    """Views [h, w, 3] of the images in a packed buffer (host or device)."""
    views, off = [], 0
    for h, w in sizes.tolist():
        views.append(packed[off:off + 3 * h * w].view(h, w, 3))
        off += 3 * h * w
    return views


class DeviceResizeLoader:
    """Wraps a DataLoader that yields collate_packed batches: each batch is copied to `device` in one piece, resized there to
    (height, width) and, with imgaug, augmented in place by img_aug_batch (the reference's order: resize, then img_aug).  Yields
    (uint8 CUDA [N, 3, height, width], targets), what utils.utils.evaluation and the train loop take from TensorDataset's loader.
    Re-iterable and sized like the loader it wraps."""

    def __init__(self, loader, width, height, device, imgaug=False, rng=random):
        self.loader, self.width, self.height, self.device = loader, int(width), int(height), torch.device(device)
        self.imgaug, self.rng = imgaug, rng

    def __len__(self):
        return len(self.loader)

    def __iter__(self):
        for packed, sizes, targets in self.loader:
            d = packed.to(self.device, non_blocking=True)
            imgs = yfv2_engine.resize_u8(unpack(d, sizes), self.height, self.width)
            if self.imgaug:
                img_aug_batch(imgs, rng=self.rng, out=imgs)
            yield imgs, targets

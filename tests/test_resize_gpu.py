"""Device resize (yfv2_resize_u8, csrc/k_resize.cu, through the C ABI) bit-exact against the real cv2 goldens and the oracle, and
the device-resize input path end to end: test.py from the decoded JPEG, resize + augmentation, forward / detections, the
evaluation loader and the training launcher."""
import os
import random

import numpy as np
import pytest
import torch

import yfv2  # noqa: F401
import synth
import yfv2_engine as eng
from oracle import aug as oaug, resize as orz

pytestmark = pytest.mark.gpu


def _packed_sources(imgs, offsets_odd=True, seed=0):
    """All images in ONE device buffer at byte offsets (odd ones when offsets_odd), returned as views."""
    rs = np.random.RandomState(seed)
    offs, cur = [], 0
    for im in imgs:
        cur += int(rs.randint(0, 16)) | 1 if offsets_odd else 0
        offs.append(cur)
        cur += im.size
    buf = np.zeros(cur + 16, np.uint8)
    for im, o in zip(imgs, offs):
        buf[o:o + im.size] = im.reshape(-1)
    d = torch.from_numpy(buf).cuda()
    return [d[o:o + im.size].view(im.shape) for im, o in zip(imgs, offs)], d


def test_bit_exact_against_cv2_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "resize_cases.npz"))
    for i, (seed, h, w, H, W) in enumerate(g["cases"]):
        src = torch.from_numpy(orz.noise_image(int(seed), int(h), int(w))).cuda()
        got = eng.resize_u8([src], int(H), int(W)).cpu().numpy()
        assert orz.matches_golden(g, i, got[0].transpose(1, 2, 0)), (i, h, w, H, W)


def test_ragged_batch_across_launches_against_oracle():
    """300 images (the C ABI splits launches at 256) of mixed up / down scales, 1-pixel and thin sources, all packed into one
    buffer at odd byte offsets."""
    rs = np.random.RandomState(11)
    sizes = [(1, 1), (1, 500), (500, 1), (2, 3), (480, 640), (640, 480)]
    sizes += [(int(rs.randint(1, 700)), int(rs.randint(1, 700))) for _ in range(300 - len(sizes))]
    imgs = [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in sizes]
    views, _ = _packed_sources(imgs, seed=12)
    H, W = 96, 160
    got = eng.resize_u8(views, H, W).cpu().numpy()
    assert got.shape == (300, 3, H, W)
    for i, im in enumerate(imgs):
        assert np.array_equal(got[i], orz.resize_linear_u8(im, H, W).transpose(2, 0, 1)), (i, im.shape)


@pytest.mark.parametrize("H,W", [(640, 640), (352, 608), (608, 352), (1024, 17), (33, 1024)])
def test_large_and_non_square_destinations(H, W):
    rs = np.random.RandomState(H * 7 + W)
    imgs = [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in ((480, 640), (427, 640), (1200, 1600), (57, 91), (1, 640))]
    views, _ = _packed_sources(imgs, offsets_odd=(H % 2 == 0), seed=H)
    got = eng.resize_u8(views, H, W).cpu().numpy()
    for i, im in enumerate(imgs):
        assert np.array_equal(got[i], orz.resize_linear_u8(im, H, W).transpose(2, 0, 1)), (i, im.shape)


def test_wide_source_limit():
    rs = np.random.RandomState(5)
    im = rs.randint(0, 256, (3, 8192, 3)).astype(np.uint8)
    got = eng.resize_u8([torch.from_numpy(im).cuda()], 4, 1024).cpu().numpy()
    assert np.array_equal(got[0], orz.resize_linear_u8(im, 4, 1024).transpose(2, 0, 1))


def _modelzoo_model(golden_dir):
    import model.detector
    w = dict(np.load(os.path.join(golden_dir, "modelzoo_weights.npz")))
    m = model.detector.Detector(80, 3, True).cuda()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    return m.eval()


def test_test_py_from_the_decoded_jpeg(golden_dir):
    """test.py:33-50 with the resize on the device: the network input equals the stored cv2 one bit for bit, and the modelzoo
    weights give the known answers (img/000139_result.png: person .87, bicycle .46, person .32; 000004: nine cars)."""
    import utils.utils as uu
    g = np.load(os.path.join(golden_dir, "resize_images.npz"))
    m_u8 = np.load(os.path.join(golden_dir, "images_modelzoo.npz"))
    model_ = _modelzoo_model(golden_dir)
    cfg = synth.coco_cfg(352, 352)
    for name in ("000139", "000004"):
        x = eng.resize_u8([torch.from_numpy(g["img_" + name]).cuda()], 352, 352)
        assert np.array_equal(x.cpu().numpy(), m_u8[name + "_u8"]), name
        with torch.no_grad():
            preds = model_(x.float() / 255.0)
        rows = uu.non_max_suppression(uu.handel_preds(preds, cfg, "cuda"), conf_thres=0.3, iou_thres=0.4)[0].numpy()
        if name == "000139":
            assert [(int(r[5]), "%.2f" % r[4]) for r in rows] == [(0, "0.87"), (1, "0.46"), (0, "0.32")]
        else:
            assert ["%.2f" % r[4] for r in rows] == ["0.87", "0.85", "0.76", "0.75", "0.68", "0.60", "0.56", "0.47", "0.33"]
            assert all(int(r[5]) == 2 for r in rows)


def test_resize_then_augmentation_matches_oracle():
    import utils.device_aug as da
    rs = np.random.RandomState(21)
    imgs = [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in ((480, 640), (333, 500), (24, 31), (700, 90))]
    views, _ = _packed_sources(imgs, seed=22)
    x = eng.resize_u8(views, 352, 352)
    da.img_aug_batch(x, rng=random.Random(7), out=x)
    r = random.Random(7)
    for i, im in enumerate(imgs):
        a, b = r.uniform(0.25, 1.75), r.uniform(0.25, 1.75)                 # the order img_aug_batch draws them
        want = oaug.contrast_and_brightness(orz.resize_linear_u8(im, 352, 352), a, b).transpose(2, 0, 1)
        assert np.array_equal(x[i].cpu().numpy(), want), i


def test_heads_and_detections_equal_those_of_the_oracle_resized_batch(golden_dir):
    import utils.utils as uu
    g = np.load(os.path.join(golden_dir, "resize_images.npz"))
    rs = np.random.RandomState(31)
    imgs = [g["img_000139"], g["img_000004"]] + [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in ((480, 640), (427, 640))]
    views, _ = _packed_sources(imgs, seed=32)
    dev_x = eng.resize_u8(views, 352, 352)
    host_x = torch.from_numpy(orz.resize_to_nchw(imgs, 352, 352)).cuda()
    assert torch.equal(dev_x, host_x)
    model_ = _modelzoo_model(golden_dir)
    cfg = synth.coco_cfg(352, 352)
    with torch.no_grad():
        pa, pb = model_(dev_x), model_(host_x)
    for a, b in zip(pa, pb):
        assert torch.equal(a, b)
    for a, b in zip(uu.detect(pa, cfg, 0.001, 0.4), uu.detect(pb, cfg, 0.001, 0.4)):
        assert torch.equal(a, b)


class _InMemoryRaw(torch.utils.data.Dataset):
    def __init__(self, items):
        self.items = items

    def __len__(self):
        return len(self.items)

    def __getitem__(self, i):
        img, lab = self.items[i]
        return torch.from_numpy(img), lab.clone()


def test_device_resize_loader_feeds_evaluation_like_the_host_resized_loader(golden_dir):
    import train_dist
    import utils.device_aug as da
    import utils.utils as uu
    g = np.load(os.path.join(golden_dir, "resize_images.npz"))
    rs = np.random.RandomState(41)
    imgs = [g["img_000139"], g["img_000004"]] + [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in ((480, 640), (375, 500), (64, 96))]
    labels = [synth.make_targets(42 + i, 1) for i in range(len(imgs))]
    raw = _InMemoryRaw(list(zip(imgs, labels)))
    host = [(torch.from_numpy(orz.resize_linear_u8(im, 352, 352).transpose(2, 0, 1).copy()), lab.clone()) for im, lab in zip(imgs, labels)]
    cfg = synth.coco_cfg(352, 352)
    model_ = _modelzoo_model(golden_dir)
    dl = torch.utils.data.DataLoader(raw, batch_size=2, shuffle=False, collate_fn=da.collate_packed, num_workers=0, pin_memory=True)
    dev_loader = da.DeviceResizeLoader(dl, cfg["width"], cfg["height"], "cuda")
    host_loader = torch.utils.data.DataLoader(host, batch_size=2, shuffle=False, collate_fn=train_dist.collate_fn, num_workers=0,
                                              pin_memory=True)
    assert len(dev_loader) == len(host_loader) == 3
    for (a, ta), (b, tb) in zip(dev_loader, host_loader):
        assert a.is_cuda and a.dtype == torch.uint8 and torch.equal(a.cpu(), b) and torch.equal(ta, tb)
    for conf in (0.01, 0.3):
        got = uu.evaluation(dev_loader, cfg, model_, "cuda", conf)
        want = uu.evaluation(host_loader, cfg, model_, "cuda", conf)
        assert got is not None
        np.testing.assert_array_equal(np.array(got), np.array(want))


DATA = ("[name]\nmodel_name=coco\n\n[train-configure]\nepochs=1\nsteps=150,250\nbatch_size=8\nsubdivisions=2\nlearning_rate=0.001\n\n"
        "[model-configure]\npre_weights=None\nclasses=80\nwidth=352\nheight=352\nanchor_num=3\n"
        "anchors=12.64,19.39, 37.88,51.48, 55.71,138.31, 126.91,78.23, 131.57,214.55, 279.92,258.87\n\n"
        "[data-configure]\ntrain=/nonexistent/train.txt\nval=/nonexistent/val.txt\nnames=/nonexistent/coco.names\n")


@pytest.mark.parametrize("extra", [[], ["--device-aug"]])
def test_launcher_with_device_resize(tmp_path, monkeypatch, extra):
    import train_dist
    data = tmp_path / "coco.data"
    data.write_text(DATA)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    net = train_dist.main(["--data", str(data), "--synthetic", "8", "--device-resize", "--max-iters", "2"] + extra)
    assert all(torch.isfinite(p).all() for p in net.parameters())

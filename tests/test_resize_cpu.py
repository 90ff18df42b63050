"""The resize restatement (oracle/resize.py) against outputs of the real cv2.resize (tests/golden/resize_cases.npz, and live cv2
where it is installed), the argument checks of yfv2_resize_u8 (no GPU needed: nothing is launched for a bad argument) and the
host side of the device-resize data path (label parsing, batch packing)."""
import ctypes
import os

import numpy as np
import pytest
import torch

import yfv2  # noqa: F401
from oracle import resize as orz


def test_oracle_matches_cv2_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "resize_cases.npz"))
    assert str(g["cv2_version"]).startswith("4.")
    assert sum(("out_%d" % i) in g for i in range(len(g["cases"]))) >= 10            # most cases are stored byte for byte
    for i, (seed, h, w, H, W) in enumerate(g["cases"]):
        got = orz.resize_linear_u8(orz.noise_image(int(seed), int(h), int(w)), int(H), int(W))
        assert orz.matches_golden(g, i, got), (i, h, w, H, W)


def test_oracle_reproduces_the_model_inputs_of_the_bundled_images(golden_dir):
    """test.py:34-37 from the decoded JPEGs: resize + transpose give the stored network inputs of images_modelzoo.npz."""
    g = np.load(os.path.join(golden_dir, "resize_images.npz"))
    m = np.load(os.path.join(golden_dir, "images_modelzoo.npz"))
    for name in ("000139", "000004"):
        assert np.array_equal(orz.resize_to_nchw([g["img_" + name]], 352, 352), m[name + "_u8"]), name


def test_oracle_matches_live_cv2_on_random_sizes():
    cv2 = pytest.importorskip("cv2")
    rs = np.random.RandomState(2024)
    for k in range(200):
        h, w = int(rs.randint(1, 600)), int(rs.randint(1, 600))
        if k % 4 == 0:                                           # exact integer downscales (OpenCV's INTER_AREA shortcut)
            f = int(rs.randint(2, 5))
            H, W = max(1, h // f), max(1, w // f)
            h, w = H * f, W * f
        else:
            H, W = int(rs.randint(1, 400)), int(rs.randint(1, 400))
        img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        want = cv2.resize(img, (W, H), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(orz.resize_linear_u8(img, H, W), want), (h, w, H, W)


def test_resize_entry_point_validates_before_touching_the_device():
    import yfv2_engine
    lib = yfv2_engine.lib()
    fake = 1 << 40                                                 # never dereferenced: every call below is rejected first

    def call(ptrs, hw, N, H, W, out):
        src = (ctypes.c_void_p * max(len(ptrs), 1))(*ptrs) if ptrs is not None else None
        shw = (ctypes.c_int * max(len(hw), 1))(*hw) if hw is not None else None
        rc = lib.yfv2_resize_u8(src, shw, N, H, W, ctypes.c_void_p(out) if out else None, None)
        return rc, lib.yfv2_last_error()

    out = fake + (1 << 30)
    bad_inval = [
        (None, [10, 10], 1, 8, 8, out),                            # null source array
        ([fake], None, 1, 8, 8, out),                              # null size array
        ([fake], [10, 10], 1, 8, 8, 0),                            # null output
        ([fake], [10, 10], 0, 8, 8, out),                          # N = 0
        ([fake], [10, 10], -3, 8, 8, out),
        ([fake], [0, 10], 1, 8, 8, out),                           # empty source
        ([fake], [10, -1], 1, 8, 8, out),
        ([fake], [10, 10], 1, 0, 8, out),                          # empty destination
        ([fake], [10, 10], 1, 8, -2, out),
        ([fake, 0], [10, 10, 10, 10], 2, 8, 8, out),               # one null source pointer
        ([fake, out + 100], [10, 10, 10, 10], 2, 8, 8, out),       # a source inside the output
        ([out - 10], [10, 10], 1, 8, 8, out),                      # a source running into the output
    ]
    for args in bad_inval:
        rc, msg = call(*args)
        assert rc == -1 and msg and b"resize_u8" in msg, (args, rc, msg)
    bad_unsupported = [
        ([fake], [8193, 10], 1, 8, 8, out),                        # above YFV2_RESIZE_MAX_SRC
        ([fake], [10, 8193], 1, 8, 8, out),
        ([fake], [10, 10], 1, 1025, 8, out),                       # above YFV2_RESIZE_MAX_DST
        ([fake], [10, 10], 1, 8, 1025, out),
    ]
    for args in bad_unsupported:
        rc, msg = call(*args)
        assert rc == -3 and msg and b"resize_u8" in msg, (args, rc, msg)
    txt = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "yfv2.h")).read()
    assert "#define YFV2_RESIZE_MAX_SRC 8192" in txt and "#define YFV2_RESIZE_MAX_DST 1024" in txt


def test_darknet_labels_and_packed_batches(tmp_path):
    import utils.device_aug as da
    p = tmp_path / "a.b.txt"
    p.write_text("3 0.5 0.25 0.1 0.2\n\n17 0.1 0.9 0.05 0.05\n")
    rows = da.read_darknet_labels(str(p))
    assert rows.dtype == torch.float32 and rows.tolist() == torch.tensor(
        [[0, 3, 0.5, 0.25, 0.1, 0.2], [0, 17, 0.1, 0.9, 0.05, 0.05]], dtype=torch.float32).tolist()
    (tmp_path / "empty.txt").write_text("")
    assert tuple(da.read_darknet_labels(str(tmp_path / "empty.txt")).shape) == (0, 6)
    with pytest.raises(Exception):
        da.read_darknet_labels(str(tmp_path / "missing.txt"))
    assert da.label_path_for("/d/x.y/img.jpg") == "/d/x.txt"          # the reference's rule: up to the first '.'
    g = torch.Generator().manual_seed(3)
    imgs = [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8) for h, w in ((5, 7), (1, 1), (13, 2))]
    labels = [torch.ones((2, 6)), torch.zeros((0, 6)), torch.ones((1, 6))]
    packed, sizes, targets = da.collate_packed(list(zip(imgs, labels)))
    assert packed.dtype == torch.uint8 and packed.dim() == 1 and packed.numel() == sum(i.numel() for i in imgs)
    assert sizes.tolist() == [[5, 7], [1, 1], [13, 2]]
    assert targets[:, 0].tolist() == [0, 0, 2]
    for a, b in zip(da.unpack(packed, sizes), imgs):
        assert torch.equal(a, b)

"""CPU restatement (test infrastructure) of the resize that starts every input path of the reference, utils/datasets.py:106-111
and test.py:34-37:

    img = cv2.resize(cv2.imread(path), (W, H), interpolation=cv2.INTER_LINEAR)

OpenCV is a third-party dependency of the reference, not part of it (the goldens record the version that made them).  For
uint8 images its INTER_LINEAR is fixed-point, per channel, with INTER_RESIZE_COEF_SCALE = 2048:
  columns  fx = fl32((dx + 0.5) * scale_x - 0.5) with scale_x = 1 / (W / w) in double; sx = floor(fx), fx -= sx; sx < 0 or
           sx >= w - 1 clamp sx to the edge and set fx = 0; a0 = rint((1 - fx) * 2048), a1 = rint(fx * 2048) in fp32
  rows     the same sy, fy, b0, b1, but fy is NOT clamped: only the row indices are (r0 = clamp(sy), r1 = clamp(sy + 1))
  pass 1   T[r][dx] = src[r][sx] * a0 + src[r][min(sx + 1, w - 1)] * a1                       (int32)
  pass 2   v = (((T[r0] >> 4) * b0) >> 16) + (((T[r1] >> 4) * b1) >> 16);  out = saturate_u8((v + 2) >> 2)
Pass 2 is the vectorised form OpenCV uses for every byte; the textbook (S0*b0 + S1*b1 + 2^21) >> 22 differs by 1 in about one
byte of eight.  Exact integer downscales, where OpenCV switches to INTER_AREA internally, give the same bytes.  Pinned to
outputs of the real cv2.resize in tests/golden/resize_cases.npz (tests/golden/make_golden_resize.py)."""
import numpy as np

COEF_SCALE = 2048


def _axis(dst, src):
    """Source index and fractional weight of every destination coordinate, as (index int64, frac fp32)."""
    scale = 1.0 / (float(dst) / float(src))                                          # double, like OpenCV
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    return s.astype(np.int64), f


def _coef(f):
    one = np.float32(1.0)
    scale = np.float32(COEF_SCALE)
    return np.rint((one - f) * scale).astype(np.int32), np.rint(f * scale).astype(np.int32)


def tables(h, w, H, W):
    """(sx0, sx1, a0, a1) over the W columns and (r0, r1, b0, b1) over the H rows."""
    sx, fx = _axis(W, w)
    fx = np.where((sx < 0) | (sx >= w - 1), np.float32(0), fx).astype(np.float32)
    sx = np.clip(sx, 0, w - 1)
    a0, a1 = _coef(fx)
    sy, fy = _axis(H, h)                                                             # fy unclamped
    b0, b1 = _coef(fy)
    return (sx, np.minimum(sx + 1, w - 1), a0, a1), (np.clip(sy, 0, h - 1), np.clip(sy + 1, 0, h - 1), b0, b1)


def resize_linear_u8(img, height, width):
    """cv2.resize(img, (width, height), interpolation=cv2.INTER_LINEAR) for an HWC uint8 image (any channel count)."""
    img = np.asarray(img, dtype=np.uint8)
    squeeze = img.ndim == 2
    if squeeze:
        img = img[:, :, None]
    h, w = img.shape[:2]
    (sx0, sx1, a0, a1), (r0, r1, b0, b1) = tables(h, w, height, width)
    rows = np.unique(np.concatenate([r0, r1]))                                       # rows in between are never read
    src = img[rows].astype(np.int32)
    t = src[:, sx0] * a0[None, :, None] + src[:, sx1] * a1[None, :, None]            # pass 1: [rows, W, C]
    pos = np.searchsorted(rows, np.arange(h)) if rows.size else rows
    t0, t1 = t[pos[r0]], t[pos[r1]]
    v = (((t0 >> 4) * b0[:, None, None]) >> 16) + (((t1 >> 4) * b1[:, None, None]) >> 16)
    out = np.clip((v + 2) >> 2, 0, 255).astype(np.uint8)
    return out[:, :, 0] if squeeze else out


def resize_to_nchw(images, height, width):
    """What yfv2_resize_u8 writes: the [N,3,H,W] uint8 batch of the resized HWC images, channel order kept."""
    return np.stack([resize_linear_u8(im, height, width).transpose(2, 0, 1) for im in images])


def noise_image(seed, h, w):
    """The seeded HWC uint8 noise sources of tests/golden/resize_cases.npz (only their seeds and sizes are stored)."""
    return np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)


def digest(img):
    """SHA-256 of an image's bytes (C order) as uint8[32]: how resize_cases.npz pins the cv2 outputs too large to store."""
    import hashlib
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(img, dtype=np.uint8).tobytes()).digest(), np.uint8).copy()


def matches_golden(g, i, img):
    """True when the HWC image equals case i of resize_cases.npz: byte for byte (`out_<i>`) or by digest (`sha256_<i>`)."""
    if "out_%d" % i in g:
        return np.array_equal(img, g["out_%d" % i])
    return np.array_equal(digest(img), g["sha256_%d" % i])

"""Golden vectors for the deploy post-process (SURVEY 8f.4): outputs of the REFERENCE's own C++ (sample/ncnn/src/yolo-fastestv2.cpp
predHandle + nmsHandle, compiled in place by `make -C oracle ref` against stub ncnn/OpenCV headers) on export_onnx head tensors.
Writes ncnn_post.npz and ncnn_post_fresh.npz (same layout, other seeds and shape).

Run where the reference checkout is available (oracle/Makefile REF):  python tests/golden/make_golden_ncnn.py
Inputs are stored in the .npz (not regenerated) so the fixture does not depend on the host's exp()/sigmoid code paths.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import synth  # noqa: E402

subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], check=True, capture_output=True)
ref = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libncnn_post_ref.so"))
ref.ncnn_ref_detect.restype = ctypes.c_int
ref.ncnn_ref_detect.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
ref.ncnn_ref_configure.restype = None
ref.ncnn_ref_configure.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p]
COCO = np.array([12.64, 19.39, 37.88, 51.48, 55.71, 138.31, 126.91, 78.23, 131.57, 214.55, 279.92, 258.87], np.float32)


def export_heads(preds):
    """model/detector.py:33-44 on six logit tensors -> two [N,h,w,5A+C] arrays."""
    outs = []
    for lv in range(2):
        reg, obj, cls = preds[3 * lv], preds[3 * lv + 1], preds[3 * lv + 2]
        o = torch.cat((reg.sigmoid(), obj.sigmoid(), torch.softmax(cls, dim=1)), 1).permute(0, 2, 3, 1)
        outs.append(o.contiguous().numpy())
    return outs


def run_ref(o2, o3, A, C, in_w, in_h, anchors, thresh, nms, src_w, src_h):
    ref.ncnn_ref_configure(A, C, in_w, in_h, nms, np.ascontiguousarray(anchors, np.float32).ctypes.data)
    cap = A * (o2.shape[0] * o2.shape[1] + o3.shape[0] * o3.shape[1])
    boxes = np.zeros((cap, 4), np.int32); scores = np.zeros(cap, np.float32); cates = np.zeros(cap, np.int32)
    n = ref.ncnn_ref_detect(o2.ctypes.data, o2.shape[0], o2.shape[1], o3.ctypes.data, o3.shape[0], o3.shape[1], o2.shape[2], src_w, src_h,
                            thresh, cap, boxes.ctypes.data, scores.ctypes.data, cates.ctypes.data)
    return boxes[:n].copy(), scores[:n].copy(), cates[:n].copy()


def no_ties(o2, o3, A, thresh):
    sc = []
    for o in (o2, o3):
        v = o.reshape(-1, o.shape[-1])
        for b in range(A):
            sc.append((v[:, 5 * A:] * v[:, 4 * A + b:4 * A + b + 1]).max(1))
    sc = np.concatenate(sc)
    sc = sc[sc > thresh]
    return len(np.unique(sc)) == len(sc)


def save(fname, cases):
    out = {}
    for (name, o2, o3, A, C, iw, ih, anc, thr, nms, sw, sh) in cases:
        assert no_ties(o2, o3, A, thr), name
        b, s, c = run_ref(np.ascontiguousarray(o2), np.ascontiguousarray(o3), A, C, iw, ih, anc, thr, nms, sw, sh)
        print(name, "kept", len(s), "top", s[:3], c[:3])
        out[name + "_out2"] = o2; out[name + "_out3"] = o3
        out[name + "_params"] = np.array([A, C, iw, ih, sw, sh], np.int32)
        out[name + "_fparams"] = np.array([thr, nms], np.float32)
        out[name + "_anchors"] = anc
        out[name + "_boxes"] = b; out[name + "_scores"] = s; out[name + "_cates"] = c
    out["names"] = np.array([c[0] for c in cases])
    np.savez_compressed(os.path.join(HERE, fname), **out)
    print("wrote", os.path.join(HERE, fname), os.path.getsize(os.path.join(HERE, fname)), "bytes")


cases = []
zoo = np.load(os.path.join(HERE, "images_modelzoo.npz"))
# 1-2: the bundled images through the modelzoo weights (352x352), the sample's defaults (thresh 0.3, NMS 0.25) and a low threshold;
#      source sizes of the real files (img/000139.jpg 640x426, img/000004.jpg 500x406): scaleW/scaleH != 1
for name, (sw, sh), thr in (("000139", (640, 426), 0.3), ("000004", (500, 406), 0.05)):
    preds = [torch.from_numpy(zoo["%s_pred%d" % (name, i)]) for i in range(6)]
    o2, o3 = export_heads(preds)
    cases.append((name, o2[0], o3[0], 3, 80, 352, 352, COCO, thr, 0.25, sw, sh))
# 3: dense synthetic logits, few dominant classes (same-class overlaps -> suppression), non-square input, scale 1
p = list(synth.make_head_logits(31, 1, 96, 128))
for i in (2, 5):
    p[i][:, :3] += 6.0
o2, o3 = export_heads(p)
cases.append(("dense96x128", o2[0], o3[0], 3, 80, 128, 96, COCO, 0.001, 0.25, 128, 96))
# 4: other shape: 2 anchors, 5 classes, 256x320 input, different NMS threshold and anchors, up-scaling
p = list(synth.make_head_logits(32, 1, 320, 256, classes=5, anchor_num=2, obj_mean=-1.0))
o2, o3 = export_heads(p)
anc = np.array([10, 14, 40, 60, 90, 70, 200, 180], np.float32)
cases.append(("a2c5_320x256", o2[0], o3[0], 2, 5, 256, 320, anc, 0.05, 0.45, 1024, 960))
save("ncnn_post.npz", cases)

# ncnn_post_fresh.npz: seeds that ncnn_post.npz does not use, at 224x160 input, 3 anchors, 80 classes, two dominant classes,
# thresh 0.01, NMS 0.3, source 448x320 (scale 2).  Three seeds keep the fixture small (~190 KB; the inputs are incompressible).
fresh = []
for seed in (40, 41, 42):
    p = list(synth.make_head_logits(seed, 1, 160, 224, obj_mean=-0.5))
    for i in (2, 5):
        p[i][:, :2] += 5.0
    o2, o3 = export_heads(p)
    fresh.append(("seed%d_224x160" % seed, o2[0], o3[0], 3, 80, 224, 160, COCO, 0.01, 0.3, 448, 320))
save("ncnn_post_fresh.npz", fresh)

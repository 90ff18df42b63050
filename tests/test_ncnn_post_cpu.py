"""CPU: oracle/ncnn_post.c (restatement of the ncnn sample's decode + per-class NMS, sample/ncnn/src/yolo-fastestv2.cpp:58-183)
against tests/golden/ncnn_post.npz and ncnn_post_fresh.npz, which hold outputs of the reference's own C++ compiled in place
(make_golden_ncnn.py)."""
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def cases(fname="ncnn_post.npz"):
    g = np.load(os.path.join(HERE, "golden", fname))
    for name in g["names"]:
        name = str(name)
        A, C, iw, ih, sw, sh = [int(v) for v in g[name + "_params"]]
        thr, nms = [float(v) for v in g[name + "_fparams"]]
        yield dict(name=name, out2=g[name + "_out2"], out3=g[name + "_out3"], A=A, C=C, iw=iw, ih=ih, sw=sw, sh=sh, thr=np.float32(thr),
                   nms=np.float32(nms), anchors=g[name + "_anchors"], boxes=g[name + "_boxes"], scores=g[name + "_scores"], cates=g[name + "_cates"])


def check_case(c):
    from oracle import ncnn_post as onp
    scale_w, scale_h = np.float32(c["sw"]) / np.float32(c["iw"]), np.float32(c["sh"]) / np.float32(c["ih"])      # .cpp:189-190 (float division)
    b, s, k = onp.ncnn_post(c["out2"], c["out3"], c["A"], c["C"], c["iw"], c["ih"], c["anchors"], c["thr"], c["nms"], scale_w, scale_h)
    assert len(s) == len(c["scores"]) > 0
    assert np.array_equal(b, c["boxes"]) and np.array_equal(k, c["cates"])
    assert np.array_equal(s.view(np.uint32), c["scores"].view(np.uint32))


@pytest.mark.parametrize("c", list(cases()), ids=lambda c: c["name"])
def test_oracle_matches_reference_cpp(c):
    check_case(c)


def test_known_answers_of_the_bundled_image():
    # img/000139_result.png: person .87, bicycle .46 -- the deploy path finds the same three objects as test.py
    c = [c for c in cases() if c["name"] == "000139"][0]
    assert [int(v) for v in c["cates"]] == [0, 1, 0]
    assert [round(float(v), 2) for v in c["scores"]] == [0.87, 0.46, 0.32]


def test_oracle_matches_live_reference_on_fresh_seeds():
    """Seeds, input shape (224x160), thresholds and source scale that ncnn_post.npz does not cover; the reference's outputs on them
    are stored in ncnn_post_fresh.npz (regenerate with make_golden_ncnn.py where the reference checkout is available)."""
    from oracle import ncnn_post as onp
    fresh = list(cases("ncnn_post_fresh.npz"))
    assert len(fresh) == 3
    for c in fresh:
        assert (c["A"], c["C"], c["iw"], c["ih"], c["sw"], c["sh"]) == (3, 80, 224, 160, 448, 320)
        assert c["out2"].shape == (10, 14, 95) and c["out3"].shape == (5, 7, 95)
        assert np.array_equal(c["anchors"], onp.ANCHORS_COCO)
        check_case(c)

"""CPU-side checks: the C-ABI library builds/loads and exports every symbol include/yfv2.h declares,
the Python mirror keeps the reference's module tree and config surface, and the product path refuses
to run without CUDA (no fallback)."""
import ctypes
import json
import os
import re

import pytest
import torch

import yfv2  # noqa: F401  (registers the package dir)
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "yfv2.h")).read()
    return sorted(set(re.findall(r"YFV2_API[^;]*?\b(yfv2_\w+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import yfv2_engine
    lib = yfv2_engine.lib()
    syms = header_symbols()
    assert len(syms) >= 16
    for s in syms:
        assert hasattr(lib, s), s
        assert s in yfv2_engine.PROTOTYPES, "ctypes prototype missing for " + s
    assert lib.yfv2_abi_version() == 1


def test_bad_arguments_are_reported_not_crashed():
    import yfv2_engine
    lib = yfv2_engine.lib()
    h = ctypes.c_void_p()
    assert lib.yfv2_plan_create(ctypes.byref(h), 0, 1, 100, 352, 3, 80, 0) == -1      # H not a multiple of 32
    assert b"multiples of 32" in lib.yfv2_last_error()
    assert lib.yfv2_plan_create(ctypes.byref(h), 0, 2, 64, 96, 3, 80, 0) == 0         # plans are host-only objects
    nb = ctypes.c_size_t()
    assert lib.yfv2_plan_workspace_bytes(h, ctypes.byref(nb)) == 0 and nb.value > 0
    assert lib.yfv2_plan_packed_bytes(h, ctypes.byref(nb)) == 0 and nb.value > 243095 * 4
    n = ctypes.c_int()
    assert lib.yfv2_plan_forward_launches(h, ctypes.byref(n)) == 0 and n.value == 14      # 24 fused stages; the stride-1 blocks of each stage chain into one launch
    assert lib.yfv2_plan_destroy(h) == 0


def test_state_dict_matches_reference_keys(golden_dir):
    import model.detector as det
    m = det.Detector(80, 3, True)
    ref = json.load(open(os.path.join(golden_dir, "statedict_keys.json")))
    got = [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()]
    assert got == ref
    assert len(list(m.parameters())) == 225 and sum(p.numel() for p in m.parameters()) == 243095
    m.load_state_dict(synth.make_state_dict(3), strict=True)
    w = dict(__import__("numpy").load(os.path.join(golden_dir, "modelzoo_weights.npz")))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()}, strict=True)       # test.py:28 contract


def test_no_cpu_fallback():
    import model.detector as det
    m = det.Detector(80, 3, True).eval()
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError):
        m.backbone(torch.zeros(1, 3, 64, 64))


def test_load_datafile(tmp_path):
    import utils.utils as uu
    p = tmp_path / "x.data"
    p.write_text("[name]\nmodel_name=coco\n\n[train-configure]\nepochs=300\nsteps=150,250\nbatch_size=128\n"
                 "subdivisions=1\nlearning_rate=0.001\n\n[model-configure]\npre_weights=None\nclasses=80\nwidth=352\n"
                 "height=352\nanchor_num=3\nanchors=12.64,19.39, 37.88,51.48, 55.71,138.31, 126.91,78.23, 131.57,214.55, 279.92,258.87\n"
                 "\n[data-configure]\ntrain=/a/train.txt\nval=/a/val.txt\nnames=./data/coco.names\nbogus=1\n")
    cfg = uu.load_datafile(str(p))
    assert cfg["anchors"] == synth.COCO_ANCHORS and cfg["steps"] == [150.0, 250.0]
    assert cfg["pre_weights"] == "None" and cfg["classes"] == 80 and cfg["learning_rate"] == 0.001
    assert (cfg["width"], cfg["height"], cfg["anchor_num"], cfg["batch_size"]) == (352, 352, 3, 128)
    assert set(cfg) == {"model_name", "epochs", "steps", "batch_size", "subdivisions", "learning_rate", "pre_weights",
                        "classes", "width", "height", "anchor_num", "anchors", "val", "train", "names"}


def test_overlay_resolves_out_of_scope_names_from_the_reference(tmp_path, golden_dir):
    """With a reference checkout behind the mirror on sys.path, utils.datasets and the utils.utils names the mirror does not define
    come from the reference while the hot-path functions stay ours (what train.py / evaluation.py need to run unchanged).  The
    checkout is a stub with the reference's layout whose modules define the public names the real ones do
    (golden/reference_names.json, make_golden_names.py)."""
    import subprocess, sys as _sys, textwrap
    names = json.load(open(os.path.join(golden_dir, "reference_names.json")))
    ref = tmp_path / "reference"
    for d in ("utils", "model"):
        (ref / d).mkdir(parents=True)
    for rel, defined in names.items():
        (ref / rel).write_text("".join("def %s(*a, **k):\n    return 'reference'\n" % n for n in defined))
    for rel in ("utils/loss.py", "model/detector.py"):              # the mirror must shadow these
        (ref / rel).write_text("raise ImportError('the reference module was imported instead of the mirror')\n")
    code = textwrap.dedent("""
        import sys
        mirror, ref, utils_names, dataset_names = %r, %r, %r, %r
        sys.path.insert(0, ref); sys.path.insert(0, mirror)
        import utils.utils as uu, utils.datasets as ud, utils.loss as ul, model.detector as md
        assert uu.__file__.startswith(mirror) and ul.__file__.startswith(mirror) and md.__file__.startswith(mirror)
        assert ud.__file__.startswith(ref) and all(getattr(ud, n)() == "reference" for n in dataset_names)
        src = {n: getattr(uu, n).__module__ for n in utils_names}
        assert src.pop("make_grid") == "_yfv2_reference_utils", "make_grid not taken from the reference"
        assert set(src.values()) == {"utils.utils"}, src          # every other name the reference defines, the mirror defines itself
        assert callable(uu.evaluation) and uu.evaluation.__globals__["non_max_suppression"] is uu.non_max_suppression
        print("ok")
    """ % (os.path.join(ROOT, "yolo-fastestv2_b200"), str(ref), names["utils/utils.py"], names["utils/datasets.py"]))
    r = subprocess.run([_sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_header_is_plain_c_and_links_from_a_c_program(tmp_path):
    """The boundary is a C ABI: include/yfv2.h must compile as C99 (-pedantic) and a plain C program must link against libyfv2.so
    and call it (yfv2_abi_version needs no GPU)."""
    import shutil
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "abi.c"
    src.write_text('#include "yfv2.h"\n#include <stdio.h>\nint main(void) { printf("%d\\n", yfv2_abi_version()); return yfv2_last_error() == 0; }\n')
    exe = tmp_path / "abi"
    libdir = os.path.join(root, "yolo-fastestv2_b200")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-lyfv2", "-Wl,-rpath," + libdir], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip()
    assert out == "1"


def test_plan_host_logic_over_shapes():
    """Plans are host-only objects: the launch list, the stage names and the buffer sizes must be well defined for every shape the
    reference accepts (H, W multiples of 32, any batch) and the shape limits must be reported, not crashed on."""
    import yfv2_engine
    lib = yfv2_engine.lib()
    sizes = {}
    for (N, H, W, A, C) in [(1, 32, 32, 3, 80), (1, 352, 352, 3, 80), (256, 352, 352, 3, 80), (2, 640, 640, 3, 80), (3, 96, 160, 2, 20),
                            (5, 224, 96, 3, 80), (1, 1024, 1024, 3, 80), (4, 352, 352, 1, 1)]:
        h = ctypes.c_void_p()
        assert lib.yfv2_plan_create(ctypes.byref(h), 0, N, H, W, A, C, 0) == 0, (N, H, W, A, C, lib.yfv2_last_error())
        ws, pk, n = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_int()
        assert lib.yfv2_plan_workspace_bytes(h, ctypes.byref(ws)) == 0 and ws.value > 0
        assert lib.yfv2_plan_packed_bytes(h, ctypes.byref(pk)) == 0 and pk.value > 0
        assert lib.yfv2_plan_forward_launches(h, ctypes.byref(n)) == 0 and 14 <= n.value <= 32
        names = []
        while True:
            nm = lib.yfv2_plan_stage_name(h, len(names))
            if nm is None:
                break
            names.append(nm.decode())
        assert names[0] == "stem" and any(s.startswith("stage4.3") for s in names) and len(names) >= 24
        groups = [lib.yfv2_plan_stage_group(h, i) for i in range(len(names))]
        assert groups == sorted(groups) and groups[0] == 0 and lib.yfv2_plan_stage_group(h, len(names)) == -1
        assert len(set(groups)) == n.value                           # one launch per group
        sizes[(N, H, W, A, C)] = ws.value
        assert lib.yfv2_plan_destroy(h) == 0
    assert sizes[(256, 352, 352, 3, 80)] > 100 * sizes[(1, 352, 352, 3, 80)] // 2      # the workspace scales with the batch
    assert sizes[(2, 640, 640, 3, 80)] > sizes[(1, 352, 352, 3, 80)]
    h = ctypes.c_void_p()
    for bad in [(0, 352, 352, 3, 80), (1, 352, 350, 3, 80), (1, 0, 352, 3, 80), (1, 352, 352, 0, 80), (1, 352, 352, 3, 0), (1, 352, 352, 3, 200)]:
        rc = lib.yfv2_plan_create(ctypes.byref(h), 0, *bad, 0)
        assert rc < 0 and lib.yfv2_last_error(), bad
    assert lib.yfv2_plan_create(ctypes.byref(h), 0, 1, 64, 64, 3, 80, 1) < 0          # training plans are yfv2_trainer_* objects


def test_trainer_layout_matches_the_module_parameters():
    """The native trainer's flat gradient buffer (the bucket the data-parallel step all-reduces) is laid out on the host: its
    offsets must be exactly the running sum of Detector.parameters() numels, for the reference shape and for others."""
    import model.detector as det
    import yfv2_engine
    lib = yfv2_engine.lib()
    lib.yfv2_trainer_destroy.restype = None
    for (N, H, W, A, C) in [(64, 352, 352, 3, 80), (2, 64, 96, 3, 80), (3, 96, 160, 2, 20)]:
        t = ctypes.c_void_p()
        assert lib.yfv2_trainer_create(ctypes.byref(t), 0, N, H, W, A, C) == 0, lib.yfv2_last_error()
        n, ws = ctypes.c_longlong(), ctypes.c_size_t()
        assert lib.yfv2_trainer_grad_floats(t, ctypes.byref(n)) == 0
        assert lib.yfv2_trainer_workspace_bytes(t, ctypes.byref(ws)) == 0 and ws.value > 0
        params = list(det.Detector(C, A, True).parameters())
        assert n.value == sum(p.numel() for p in params)
        off = 0
        for i, p in enumerate(params):
            o, k = ctypes.c_longlong(), ctypes.c_longlong()
            assert lib.yfv2_trainer_param_offset(t, i, ctypes.byref(o), ctypes.byref(k)) == 0
            assert (o.value, k.value) == (off, p.numel()), i
            off += p.numel()
        o, k = ctypes.c_longlong(), ctypes.c_longlong()
        assert lib.yfv2_trainer_param_offset(t, len(params), ctypes.byref(o), ctypes.byref(k)) < 0
        lib.yfv2_trainer_destroy(t)
    t = ctypes.c_void_p()
    assert lib.yfv2_trainer_create(ctypes.byref(t), 0, 2, 100, 96, 3, 80) < 0 and lib.yfv2_last_error()


def test_post_processing_entry_points_validate_before_touching_the_device():
    """Argument errors of the decode / NMS / deploy post-process calls are reported through the return code and yfv2_last_error()
    before anything is launched (so this runs without a GPU)."""
    import yfv2_engine
    lib = yfv2_engine.lib()
    six = (ctypes.c_void_p * 6)()                                    # six null head tensors
    anchors = (ctypes.c_double * 12)(*range(1, 13))
    assert lib.yfv2_decode(six, 1, 352, 352, 3, 80, anchors, None, None) < 0 and lib.yfv2_last_error()
    assert lib.yfv2_decode(six, 1, 350, 352, 3, 80, anchors, None, None) < 0 and b"32" in lib.yfv2_last_error()
    assert lib.yfv2_decode_nms(six, 1, 352, 352, 3, 80, anchors, ctypes.c_float(0.3), ctypes.c_double(0.4), None, 0, 300,
                               ctypes.c_float(4096.0), None, None, None, None, None) < 0
    assert lib.yfv2_nms(None, 1, 1815, 80, ctypes.c_float(0.3), ctypes.c_double(0.4), None, 0, 300, ctypes.c_float(4096.0),
                        None, None, None, None, None) < 0
    fa = (ctypes.c_float * 12)(*range(1, 13))
    assert lib.yfv2_ncnn_post(None, None, 1, 352, 352, 3, 80, fa, ctypes.c_float(0.3), ctypes.c_float(0.25), ctypes.c_float(1), ctypes.c_float(1),
                              10, None, None, None, None, None) < 0 and b"ncnn_post" in lib.yfv2_last_error()
    assert lib.yfv2_debug_nms_profile(None) == 0

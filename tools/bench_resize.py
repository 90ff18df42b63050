#!/usr/bin/env python
"""Device resize (yfv2_resize_u8) on a batch of 256 decoded COCO-like images -> 352x352, and the inference step that starts
from decoded images instead of pre-resized ones.  Prints one JSON line (and writes it to --out when given):
  resize      CUDA events over >= --seconds of back-to-back resizes, two alternating source batches (each larger than the
              126 MB L2); us per batch, img/s, and algorithmic bytes (source rows the interpolation reads x 3w + 3HW written) over
              time against MEASURED_PEAKS.json hbm_gbs (an algorithmic rate, not a measured DRAM counter)
  raw_step    resize + forward_u8 + fused decode/NMS, beside the pre-resized step (forward_u8 + decode/NMS) of bench.py, same run
  e2e_raw     pinned host packed decoded images in (ONE host-to-device copy per batch), pinned host detections out, 3 streams in
              flight, as bench.py's e2e leg
  parity      the first 8 resized images equal oracle/resize.py byte for byte
  gpu         card name and power limit the numbers were measured at

    python tools/bench_resize.py [--seconds 1.5] [--out bench_resize.json]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import yfv2  # noqa: E402,F401
import bench  # noqa: E402
import yfv2_engine as eng  # noqa: E402
from oracle import resize as orz  # noqa: E402

BATCH, SIDE = 256, 352
SIZES = [(480, 640), (640, 480), (427, 640), (375, 500), (333, 500)]          # (h, w), COCO-like


def make_batch(seed):
    """A packed host buffer of BATCH decoded images (sizes cycled through SIZES), their sizes and byte offsets."""
    g = torch.Generator().manual_seed(seed)
    sizes = [SIZES[(i + seed) % len(SIZES)] for i in range(BATCH)]
    offs = np.concatenate([[0], np.cumsum([3 * h * w for h, w in sizes])])
    packed = torch.randint(0, 256, (int(offs[-1]),), generator=g, dtype=torch.uint8)
    return packed, sizes, offs


def views(buf, sizes, offs):
    return [buf[int(o):int(o) + 3 * h * w].view(h, w, 3) for (h, w), o in zip(sizes, offs)]


def resize_call(buf, sizes, offs, out):
    """yfv2_resize_u8 on prepared descriptor arrays (what yfv2_engine.resize_u8 builds per call, built once here so that the timed
    loop measures the device and not Python's per-image checks)."""
    base = buf.data_ptr()
    src = (ctypes.c_void_p * len(sizes))(*[base + int(o) for o in offs[:len(sizes)]])
    hw = (ctypes.c_int * (2 * len(sizes)))(*[v for s in sizes for v in s])
    L, dst = eng.lib(), ctypes.c_void_p(out.data_ptr())

    def run(stream):
        rc = L.yfv2_resize_u8(src, hw, len(sizes), out.shape[2], out.shape[3], dst, ctypes.c_void_p(stream.cuda_stream))
        if rc:
            raise RuntimeError(L.yfv2_last_error())
    return run


def algorithmic_bytes(sizes, H=SIDE, W=SIDE):
    """Source bytes of the rows the interpolation reads (rows a large downscale skips are not counted) + the NCHW output."""
    total = 0
    for h, w in sizes:
        _, (r0, r1, _, _) = orz.tables(h, w, H, W)
        total += len(np.union1d(r0, r1)) * 3 * w + 3 * H * W
    return total


def gpu_info(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        q = "unavailable (%s)" % type(e).__name__
    return {"name": name, "power_limit_and_max_sm_clock": q}


def timed(fn, seconds, stream, warmup=5):
    """us per call of fn(i) over a window of at least `seconds`, CUDA events around the whole window."""
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn(0)
    torch.cuda.synchronize()
    reps = max(20, int(seconds / max(time.perf_counter() - t0, 1e-6)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(reps):
        fn(i)
    e1.record(stream)
    e1.synchronize()
    return 1e3 * e0.elapsed_time(e1) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.5)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    binding, _ = bench.bind_to_gpu_node(0)
    stream = torch.cuda.current_stream(dev)
    batches = [make_batch(s) for s in (1, 2)]
    dsrc = [(p.to(dev), sz, o) for p, sz, o in batches]
    x = torch.empty((BATCH, 3, SIDE, SIDE), dtype=torch.uint8, device=dev)
    calls = [resize_call(*b, x) for b in dsrc]

    # ---- resize alone ----
    def resize(i):
        calls[i % 2](stream)
    us, reps = timed(resize, args.seconds, stream)
    nbytes = [algorithmic_bytes(sz) for _, sz, _ in batches]
    peak, peak_src = bench.measured_peak()
    gbs = 0.5 * (nbytes[0] + nbytes[1]) / (us * 1e-6) / 1e9
    resize_line = {"us_per_batch": us, "img_per_s": BATCH / (us * 1e-6), "reps": reps,
                   "source_batch_mb": [round(b[0].numel() / 1e6, 1) for b in batches],
                   "algorithmic_bytes_per_batch": nbytes, "algorithmic_gbs": gbs, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
                   "share_of_hbm_peak_algorithmic": gbs / peak}

    # parity: first 8 images of the last batch resized against the oracle
    eng.resize_u8(views(*dsrc[0]), SIDE, SIDE, out=x)                     # (the public wrapper once)
    got = x[:8].cpu().numpy()
    host = views(*batches[0])
    parity = all(np.array_equal(got[i], orz.resize_linear_u8(host[i].numpy(), SIDE, SIDE).transpose(2, 0, 1)) for i in range(8))

    # ---- raw step vs pre-resized step (bench.py's step: forward_u8 + fused decode/NMS) ----
    model, _ = bench.random_state_dict()
    model = model.to(dev).eval()
    c = bench.cfg()
    plan = model._plan_for(x)
    preds = plan.alloc_preds()
    anchors = eng.anchors_array(c)
    out = torch.empty((BATCH, eng.MAX_DET, 6), dtype=torch.float32, device=dev)
    counts = torch.empty((BATCH,), dtype=torch.int32, device=dev)
    L = eng.lib()
    xs_pre = [(torch.rand(BATCH, 3, SIDE, SIDE, generator=torch.Generator().manual_seed(7 + k)) * 255).to(torch.uint8).to(dev)
              for k in range(2)]

    def detect(xin, pl, pr, o, cn, s):
        pl.forward(xin, pr)
        rc = L.yfv2_decode_nms(eng._ptr_array(pr), BATCH, SIDE, SIDE, bench.ANCHORS, bench.CLASSES, anchors, ctypes.c_float(bench.CONF),
                               ctypes.c_double(bench.IOU), None, 0, eng.MAX_DET, ctypes.c_float(eng.MAX_WH), ctypes.c_void_p(o.data_ptr()),
                               ctypes.c_void_p(cn.data_ptr()), None, None, ctypes.c_void_p(s.cuda_stream))
        if rc:
            raise RuntimeError(L.yfv2_last_error())

    def pre_step(i):
        detect(xs_pre[i % 2], plan, preds, out, counts, stream)

    def raw_step(i):
        resize(i)
        detect(x, plan, preds, out, counts, stream)
    steps = {}
    for name, fn in (("pre_resized", pre_step), ("raw", raw_step), ("pre_resized_again", pre_step), ("raw_again", raw_step)):
        us_, reps_ = timed(fn, args.seconds, stream)
        steps[name] = {"ms_per_step": us_ / 1e3, "img_per_s": BATCH / (us_ * 1e-6), "reps": reps_}

    # ---- e2e from pinned host decoded images: one packed H2D per batch, 3 streams / buffers in flight ----
    nbuf = 3
    plans = [eng.Plan(dev, BATCH, SIDE, SIDE, bench.ANCHORS, bench.CLASSES, detect_max_det=eng.MAX_DET) for _ in range(nbuf)]
    params, bn = model._weight_tensors()
    for p_ in plans:
        p_.pack(params, bn)
    hsrc = [batches[b % 2][0].pin_memory() for b in range(nbuf)]
    meta = [batches[b % 2][1:] for b in range(nbuf)]
    dbuf = [torch.empty_like(h, device=dev) for h in hsrc]
    xb = [torch.empty((BATCH, 3, SIDE, SIDE), dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    rcalls = [resize_call(dbuf[b], *meta[b], xb[b]) for b in range(nbuf)]
    pb = [p_.alloc_preds() for p_ in plans]
    ob = [torch.empty((BATCH, eng.MAX_DET, 6), dtype=torch.float32, device=dev) for _ in range(nbuf)]
    cb = [torch.empty((BATCH,), dtype=torch.int32, device=dev) for _ in range(nbuf)]
    oh = [torch.empty((BATCH, eng.MAX_DET, 6), dtype=torch.float32).pin_memory() for _ in range(nbuf)]
    ch = [torch.empty((BATCH,), dtype=torch.int32).pin_memory() for _ in range(nbuf)]
    streams = [torch.cuda.Stream(dev) for _ in range(nbuf)]

    def e2e_step(i):
        b = i % nbuf
        with torch.cuda.stream(streams[b]):
            dbuf[b].copy_(hsrc[b], non_blocking=True)
            rcalls[b](streams[b])
            detect(xb[b], plans[b], pb[b], ob[b], cb[b], streams[b])
            oh[b].copy_(ob[b], non_blocking=True)
            ch[b].copy_(cb[b], non_blocking=True)

    for i in range(6):
        e2e_step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(2 * nbuf):
        e2e_step(i)
    torch.cuda.synchronize()
    reps_e2e = max(30, int(args.seconds / ((time.perf_counter() - t0) / (2 * nbuf))))
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for st_ in streams:
        st_.wait_event(s0)
    for i in range(reps_e2e):
        e2e_step(i)
    for st_ in streams:
        ev = torch.cuda.Event()
        ev.record(st_)
        stream.wait_event(ev)
    s1.record(stream)
    s1.synchronize()
    ms = s0.elapsed_time(s1)
    e2e = {"img_per_s": BATCH * reps_e2e / (ms * 1e-3), "ms_per_batch": ms / reps_e2e, "reps": reps_e2e,
           "h2d_bytes_per_batch": [int(h.numel()) for h in hsrc[:2]],
           "d2h_bytes_per_batch": oh[0].numel() * 4 + ch[0].numel() * 4, "host_binding": binding,
           "api": "pinned packed decoded images -> one H2D copy -> yfv2_resize_u8 -> forward_u8 -> decode_nms -> pinned host, 3 streams"}

    line = {"tool": "bench_resize", "batch": BATCH, "dst": [SIDE, SIDE], "sizes": SIZES, "gpu": gpu_info(dev),
            "resize": resize_line, "step": steps, "e2e_raw": e2e, "parity_first8_vs_oracle": parity}
    txt = json.dumps(line)
    print(txt, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    if not parity:
        raise SystemExit("bench_resize: resized images differ from the oracle")


if __name__ == "__main__":
    main()

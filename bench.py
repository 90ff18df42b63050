#!/usr/bin/env python
"""bench.py — images/s of the Yolo-FastestV2 hot path (forward + decode + NMS) on B200.

Workload (BASELINE.json configs[1]): batch 256 of 352x352 synthetic images per GPU, random-init weights
(seed 1, BN running stats (0,1)), decode + NMS(conf 0.001, iou 0.4) — the regime where every one of the 1815
candidates passes the confidence filter and the 300-detection cap is hit.

  python bench.py [--gpus N --steps K --warmup W]          our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference ...                      the CPU restatement of the reference (oracle/) on host cores
  python bench.py ... --dump-outputs DIR                    also write what the last timed step computed as DIR/<name>.npy

One JSON line on stdout (rank 0).  `value` = whole-job images/s with inputs resident in HBM; `e2e` = the same
through yfv2_detect_u8_host with pinned HOST uint8 images in and pinned HOST detections out, copies inside the
timed region; `roofline` = the slowest fused kernel against the measured HBM peak; `cpu_baseline` = the oracle
port on the host cores (a bounded sample).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

BATCH, SIDE, CLASSES, ANCHORS = 256, 352, 80, 3
CONF, IOU = 0.001, 0.4
METRIC = "images/sec 352x352 fwd+decode+NMS"
UNIT_NAMES = (["stem"] + ["stage2.%d" % i for i in range(4)] + ["stage3.%d" % i for i in range(8)]
              + ["stage4.%d" % i for i in range(4)] + ["fpn.S3", "fpn.S2", "heads2.a", "heads2.b", "heads3.a", "heads3.b"])
DUMP_BYTES = 64_000_000 - 4096      # --dump-outputs: all .npy files together (headers included) stay under 64 MB


def cfg():
    import synth
    return synth.coco_cfg(SIDE, SIDE, CLASSES)


def random_state_dict():
    """Detector default PyTorch init under seed 1, BN running stats left at (0,1) (SURVEY 8d config[1])."""
    import yfv2  # noqa: F401
    import model.detector as det
    import contextlib
    torch.manual_seed(1)
    with contextlib.redirect_stdout(sys.stderr):          # the mirror prints "load param..." like the reference
        m = det.Detector(CLASSES, ANCHORS, True)
    return m, {k: v.clone() for k, v in m.state_dict().items()}


def algorithmic_bytes_per_image(H=SIDE, W=SIDE, A=ANCHORS, C=CLASSES, in_bytes=4):
    """SURVEY.md 8(d): one read of each fused unit's input + one write of its output, fp32, weights excluded.
    in_bytes: bytes per input pixel-channel (1 when the uint8 images are what sits in HBM, utils/utils.py:368)."""
    hw = lambda s: (H // s) * (W // s)
    b = [in_bytes * 3 * H * W + 4 * 24 * hw(4)]
    for st, (K, s_in, s_out, rep) in enumerate(((24, 4, 8, 4), (48, 8, 16, 8), (96, 16, 32, 4))):
        b.append(4 * (K * hw(s_in) + 2 * K * hw(s_out)))
        b += [4 * (2 * K * hw(s_out)) * 2] * (rep - 1)
    b.append(4 * (192 * hw(32) + 72 * hw(32)))
    b.append(4 * ((192 * hw(32) + 96 * hw(16)) + 72 * hw(16)))
    for s in (16, 32):
        b.append(2 * 4 * (72 * hw(s) + 72 * hw(s)))                              # first halves of both heads
        b.append(2 * 4 * (72 * hw(s) + 72 * hw(s)) + 4 * (2 * 72 + 5 * A + C) * hw(s))   # second halves + output convs
    return b


def _cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if part:
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_node(dev_index):
    """Pin this process to the CPUs of ONE NUMA node before any pinned host buffer is allocated (first touch decides where its pages
    live): the host->device feed of the e2e leg otherwise depends on which socket the scheduler happened to pick (round 1: 83 k vs
    95 k img/s on identical code; round 2: 113 k .. 139 k).  Which node feeds the GPU fastest is MEASURED (64 MB pinned buffer first
    touched under each node's affinity, a few timed H2D copies) rather than read from sysfs: on the round-2 boxes the node sysfs
    calls local to the GPU was the slower one (43 vs 52 GB/s).  Returns (description, previous affinity) or (None, None)."""
    try:
        import glob
        prev = os.sched_getaffinity(0)
        nodes = []
        for d in sorted(glob.glob("/sys/devices/system/node/node[0-9]*")):
            cpus = _cpulist(open(d + "/cpulist").read()) & prev
            if cpus:
                nodes.append((os.path.basename(d), cpus))
        if len(nodes) < 2:
            return None, None
        dev = torch.device("cuda", dev_index)
        dst = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
        best = None
        for name, cpus in nodes:
            os.sched_setaffinity(0, cpus)
            src = torch.zeros(64 << 20, dtype=torch.uint8).pin_memory()
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(6):
                dst.copy_(src, non_blocking=True)
            e1.record()
            e1.synchronize()
            gbs = 6 * (64 << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9
            del src
            if best is None or gbs > best[0]:
                best = (gbs, name, cpus)
        os.sched_setaffinity(0, best[2])
        return "bound to NUMA %s of %d (%d cpus; measured pinned H2D %.1f GB/s, the best node)" % (best[1], len(nodes), len(best[2]), best[0]), prev
    except Exception:
        try:
            os.sched_setaffinity(0, prev)
        except Exception:
            pass
        return None, None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            while not self._halt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:      # NVML missing: report nothing rather than guess
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------------------
def cpu_reference_throughput(min_seconds, batch, threads=None, steps=None, warmup=1):
    """Times the oracle port (forward + decode + NMS) on the host cores.  Returns (img/s, info).

    oneDNN on a 128-core host is SLOWER with all threads on these tiny convolutions than with a few, so the thread count
    is auto-tuned (one probe step each) and the best one is what `cores` reports."""
    from oracle import net as onet, post as opost
    import synth
    _, sd = random_state_dict()
    c = cfg()
    x = synth.make_images(1, batch, SIDE, SIDE)

    def step():
        with torch.no_grad():
            preds = onet.forward(sd, x)
        dets = opost.decode(preds, c)
        return opost.nms(dets, CONF, IOU)

    ncpu = os.cpu_count() or 1
    if threads is None:
        best, best_t = None, None
        for cand in [t for t in (8, 16, 32, 64, 128, 256) if t <= ncpu] or [ncpu]:
            torch.set_num_threads(cand)
            step()
            t0 = time.perf_counter(); step(); el = time.perf_counter() - t0
            if best is None or el < best:
                best, best_t = el, cand
            if el > 3.0 * best:
                break
        threads = best_t
    torch.set_num_threads(threads)
    for _ in range(warmup):
        step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if (steps is not None and n >= steps) or (steps is None and el >= min_seconds):
            break
    return n * batch / el, {"cores": threads, "kind": "port", "ms_per_step": 1e3 * el / n,
                            "sample": "%d step(s) of batch %d @%dx%d: oracle forward+decode+NMS(%g,%g); torch intra-op threads auto-tuned "
                                      "to %d of %d host cores, C NMS" % (n, batch, SIDE, SIDE, CONF, IOU, threads, ncpu)}


def run_reference(args, rank):
    if rank != 0:
        return
    batch = 16
    v, info = cpu_reference_throughput(0, batch, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": info["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "batch=256 352x352 inference (backbone+FPN+head+decode+NMS), random weights; "
                                   "CPU arm runs bounded steps of batch %d" % batch},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def parity_check(model, x, preds, out, counts, c, dev, n=8):
    """The bench's own weights and inputs against the oracle: six head tensors within 1e-4, decode within 1e-4, NMS rows
    bit-exact on identical decoded input, fused decode+NMS identical to decode -> NMS.  Raises on a mismatch."""
    import numpy as np
    import yfv2_engine as eng
    from oracle import net as onet, post as opost
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    xs = x[:n].cpu()
    if xs.dtype == torch.uint8:
        xs = xs.float() / 255.0                              # utils/utils.py:368
    with torch.no_grad():
        ref = onet.forward(sd, xs)
    worst = 0.0
    for i, (p_, r_) in enumerate(zip(preds, ref)):
        a, b = p_[:n].cpu().numpy(), r_.numpy()
        worst = max(worst, float(np.abs(a - b).max()))
        np.testing.assert_allclose(a, b, rtol=1e-4, atol=1e-4, err_msg="bench parity: head tensor %d" % i)
    p8 = [p_[:n].contiguous() for p_ in preds]
    dets = eng.decode(p8, c)
    np.testing.assert_allclose(dets.cpu().numpy(), opost.decode(ref, c).numpy(), rtol=1e-4, atol=1e-4, err_msg="bench parity: decode")
    got, cnt, _ = eng.nms(dets, CONF, IOU, want_idx=False)
    want = opost.nms(dets.cpu(), CONF, IOU)
    for i, w_ in enumerate(want):
        k = int(cnt[i])
        if k != w_.shape[0] or not np.array_equal(got[i, :k].cpu().numpy(), w_.numpy()):
            raise AssertionError("bench parity: NMS rows of image %d differ from the oracle" % i)
        if int(counts[i]) != k or not torch.equal(out[i, :k], got[i, :k]):
            raise AssertionError("bench parity: fused decode+NMS differs from decode -> NMS on image %d" % i)
    return {"images": n, "max_abs_err_heads": worst, "tol": 1e-4, "nms": "bit-exact vs oracle on identical decoded input",
            "fused_equals_unfused": True}


def dump_outputs(d, preds, out, counts):
    """Writes what a caller of the timed path holds after its last step, as d/<name>.npy: the six head tensors
    (reg_s16, obj_s16, cls_s16, reg_s32, obj_s32, cls_s32; float32 NCHW), the detections [N,300,6] (float32; rows past
    counts[i] are not part of the result and are written as zeros) and counts [N] (float64).  image_index.npy (float64) lists
    the batch positions written: all of them, or a fixed seeded subset when the whole batch would exceed DUMP_BYTES."""
    import numpy as np
    arrays = {}
    for lv, s in enumerate((16, 32)):
        for j, nm in enumerate(("reg", "obj", "cls")):
            arrays["%s_s%d" % (nm, s)] = preds[3 * lv + j]
    valid = torch.arange(out.shape[1], device=out.device)[None, :] < counts[:, None]
    arrays["detections"] = torch.where(valid[:, :, None], out, torch.zeros((), dtype=out.dtype, device=out.device))
    arrays["counts"] = counts.double()
    n = counts.shape[0]
    per_image = sum(a[0].numel() * a.element_size() for a in arrays.values()) + 8
    idx = torch.arange(n)
    if per_image * n > DUMP_BYTES:
        k = max(1, DUMP_BYTES // per_image)
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a[idx.to(a.device)].cpu().numpy())
    np.save(os.path.join(d, "image_index.npy"), idx.double().numpy())
    return len(idx)


# ------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import yfv2  # noqa: F401
    import yfv2_engine as eng
    import synth
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    host_binding, prev_affinity = bind_to_gpu_node(local_rank)
    model, _ = random_state_dict()
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(1 + rank)
    u8 = args.input == "u8"
    if u8:
        # what the reference's evaluation loop holds on the device (utils/utils.py:368: imgs.to(device).float() / 255.0 — the
        # uint8 batch is moved first, the conversion runs on the device; here it is fused into the stem).  Two batches are
        # alternated so that the input of a step (2 x 95 MB > the 126 MB L2) can never be served from cache.
        xs_dev = [(torch.rand(BATCH, 3, SIDE, SIDE, generator=g) * 255).to(torch.uint8).to(dev) for _ in range(2)]
    else:
        xs_dev = [torch.rand(BATCH, 3, SIDE, SIDE, generator=g).to(dev)]  # 380 MB fp32 > L2 (126 MB)
    x = xs_dev[0]
    c = cfg()
    plan = model._plan_for(x)
    preds = plan.alloc_preds()
    anchors = eng.anchors_array(c)
    import ctypes
    out = torch.empty((BATCH, eng.MAX_DET, 6), dtype=torch.float32, device=dev)
    counts = torch.empty((BATCH,), dtype=torch.int32, device=dev)
    L = eng.lib()
    stream = torch.cuda.current_stream(dev)

    it = [0]

    def step():
        plan.forward(xs_dev[it[0] % len(xs_dev)], preds)
        it[0] += 1
        rc = L.yfv2_decode_nms(eng._ptr_array(preds), BATCH, SIDE, SIDE, ANCHORS, CLASSES, anchors, ctypes.c_float(CONF),
                               ctypes.c_double(IOU), None, 0, eng.MAX_DET, ctypes.c_float(eng.MAX_WH),
                               ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(counts.data_ptr()), None, None,
                               ctypes.c_void_p(stream.cuda_stream))
        if rc:
            raise RuntimeError(L.yfv2_last_error())

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    it[0] = 0
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t.item())
    value = world * BATCH * args.steps / (ms / 1e3)
    kept = int(counts.sum().item())
    if args.dump_outputs and rank == 0:                       # before anything below reuses preds / out / counts
        k = dump_outputs(args.dump_outputs, preds, out, counts)
        print("bench.py: wrote the outputs of timed step %d (%d of %d images) to %s" % (args.steps, k, BATCH, args.dump_outputs),
              file=sys.stderr)

    # ---- parity of THIS workload (outside the timed region): first images of the step against the CPU oracle ---------
    parity = None
    if rank == 0:
        last = xs_dev[(it[0] - 1) % len(xs_dev)]             # the batch the final timed step ran on
        parity = parity_check(model, last, preds, out, counts, c, dev)

    # ---- e2e: pinned host uint8 in, pinned host detections out, double buffered on two streams ------------
    e2e = None
    try:
        nbuf = 3        # input / result buffers in flight (the H2D copy of step i+2 overlaps compute of i+1 and the D2H of i)
        plans = [eng.Plan(dev, BATCH, SIDE, SIDE, ANCHORS, CLASSES, detect_max_det=eng.MAX_DET) for _ in range(nbuf)]
        params, bn = model._weight_tensors()
        for p_ in plans:
            p_.pack(params, bn)
        xs = [(torch.rand(BATCH, 3, SIDE, SIDE, generator=g) * 255).to(torch.uint8).pin_memory() for _ in range(nbuf)]
        outs = [torch.empty((BATCH, eng.MAX_DET, 6), dtype=torch.float32).pin_memory() for _ in range(nbuf)]
        cnts = [torch.empty((BATCH,), dtype=torch.int32).pin_memory() for _ in range(nbuf)]
        streams = [torch.cuda.Stream(dev) for _ in range(nbuf)]

        def e2e_step(i):
            b = i % nbuf
            with torch.cuda.stream(streams[b]):
                plans[b].detect_u8_host(xs[b], anchors, CONF, IOU, outs[b], cnts[b])

        for i in range(max(args.warmup, 3)):
            e2e_step(i)
        barrier()
        s0 = torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for st_ in streams:
            st_.wait_event(s0)
        for i in range(args.steps):
            e2e_step(i)
        for st_ in streams:
            ev = torch.cuda.Event()
            ev.record(st_)
            stream.wait_event(ev)
        s1 = torch.cuda.Event(enable_timing=True)
        s1.record(stream)
        barrier()
        ms2 = s0.elapsed_time(s1)
        t2 = torch.tensor([ms2], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(t2, op=torch.distributed.ReduceOp.MAX)
        e2e = {"value": world * BATCH * args.steps / (float(t2.item()) / 1e3), "unit": "images/s",
               "h2d_bytes_per_step": xs[0].numel(), "d2h_bytes_per_step": outs[0].numel() * 4 + cnts[0].numel() * 4,
               "api": "yfv2_detect_u8_host (pinned uint8 NCHW in, [N,300,6]+counts out), 3 streams / buffers in flight",
               "kept_check": int(sum(int(c_.sum()) for c_ in cnts))}
        del plans
    except Exception as ex:     # never hide a failure: report it in the line
        e2e = {"value": None, "error": repr(ex)}

    # ---- per-stage timing (rank 0) -> roofline of the slowest fused kernel ------------------------------------
    roof, stages = None, None
    if rank == 0:
        peak, peak_src = measured_peak()
        bpi = algorithmic_bytes_per_image(SIDE, SIDE, in_bytes=1 if u8 else 4)
        flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)       # 256 MB > L2
        reps = max(3, min(args.steps, 10))
        plan.forward(x, preds)
        unit_bytes = dict(zip(UNIT_NAMES, bpi))
        # one timing per kernel launch: consecutive stages with the same stage_groups value are one chained launch
        groups = []
        for st, gid in enumerate(plan.stage_groups):
            if groups and groups[-1][0] == gid:
                groups[-1][2] = st + 1
            else:
                groups.append([gid, st, st + 1])
        launches = []
        for _, first, last in groups:
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                plan.forward_range(x, preds, first, last)
                b.record(stream)
                b.synchronize()
                tot += a.elapsed_time(b)
            units = []
            for n_ in plan.stage_names[first:last]:
                if n_.split("/")[0] not in units:
                    units.append(n_.split("/")[0])
            launches.append((units, 1e3 * tot / reps))
        # a fused unit of SURVEY 8(d) may be more than one launch (K=96 blocks: pw1 + dw/pw2: summed), and one launch may
        # cover several units (chained stride-1 blocks: their algorithmic bytes are summed)
        stages = []
        for units, us in launches:
            if stages and stages[-1]["_units"] == units:
                stages[-1]["us"] += us
                stages[-1]["launches"] += 1
                continue
            label = units[0] if len(units) == 1 else "%s-%s" % (units[0], units[-1].split(".")[-1])
            stages.append({"stage": label, "us": us, "launches": 1, "_units": units,
                           "alg_MB": round(sum(unit_bytes[u] for u in units) * BATCH / 1e6, 2)})
        for s_ in stages:
            gbs = s_["alg_MB"] * 1e6 / (s_["us"] * 1e-6) / 1e9
            s_["units"] = len(s_.pop("_units"))
            s_["us"] = round(s_["us"], 2)
            s_["GBps"] = round(gbs, 1)
            s_["frac"] = round(gbs / peak, 4)
        # the post-processing launch, timed the same way (not a bandwidth kernel: a greedy per-image chain; its algorithmic bytes are
        # the head tensors it reads and the [N,300,6] detections it writes)
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            rc = L.yfv2_decode_nms(eng._ptr_array(preds), BATCH, SIDE, SIDE, ANCHORS, CLASSES, anchors, ctypes.c_float(CONF),
                                   ctypes.c_double(IOU), None, 0, eng.MAX_DET, ctypes.c_float(eng.MAX_WH),
                                   ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(counts.data_ptr()), None, None,
                                   ctypes.c_void_p(stream.cuda_stream))
            b.record(stream)
            b.synchronize()
            tot += a.elapsed_time(b)
        hw_ = (SIDE // 16) ** 2 + (SIDE // 32) ** 2
        post_MB = BATCH * (4 * (5 * ANCHORS + CLASSES) * hw_ + 4 * (eng.MAX_DET * 6 + 1)) / 1e6
        post = {"stage": "decode+nms", "us": round(1e3 * tot / reps, 2), "launches": 1, "alg_MB": round(post_MB, 2), "units": 1}
        post["GBps"] = round(post_MB * 1e6 / (post["us"] * 1e-6) / 1e9, 1)
        post["frac"] = round(post["GBps"] / peak, 4)
        top = max(stages, key=lambda s: s["us"])                 # slowest launch of the NETWORK (the roofline target of north_star)
        bb = [s for s in stages if s["stage"].startswith(("stem", "stage"))]
        bb_bytes = sum(s["alg_MB"] for s in bb) * 1e6
        bb_us = sum(s["us"] for s in bb)
        traffic = None
        try:        # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture of this workload
            with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:       # regenerate: tools/ncu_traffic.py
                per = json.load(f)["per_launch_bytes"]
            traffic = per.get(top["stage"])
            for s_ in stages:
                if per.get(s_["stage"]):
                    s_["traffic_ratio"] = round(per[s_["stage"]] / (s_["alg_MB"] * 1e6), 3)
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": top["stage"], "achieved": top["GBps"], "peak": peak, "unit": "GB/s",
                "frac": top["frac"], "traffic": traffic, "algorithmic_bytes": int(top["alg_MB"] * 1e6),
                "peak_source": peak_src + " (of measured)", "timing": "CUDA events, L2 flushed before each launch",
                "backbone": {"achieved": round(bb_bytes / (bb_us * 1e-6) / 1e9, 1), "frac": round(bb_bytes / (bb_us * 1e-6) / 1e9 / peak, 4),
                             "us": round(bb_us, 1)},
                "scope": "slowest launch of the network (stem .. heads); the post-processing launch is listed in `stages` as decode+nms"}
        try:
            if per.get("decode+nms"):
                post["traffic_ratio"] = round(per["decode+nms"] / (post["alg_MB"] * 1e6), 3)
        except Exception:
            pass
        stages.append(post)
        try:        # the whole timed step against the same peak: algorithmic bytes of every launch / the step time of `value`
            step_bytes = sum(float(s_["alg_MB"]) for s_ in stages) * 1e6
            step_gbs = step_bytes / ((ms / args.steps) * 1e-3) / 1e9
            roof["step"] = {"achieved": round(step_gbs, 1), "frac": round(step_gbs / peak, 4), "algorithmic_bytes": int(step_bytes),
                            "ms": round(ms / args.steps, 4)}
        except Exception:
            pass
        del flush

    cpu = None
    if rank == 0 and world == 1 and not os.environ.get("YFV2_BENCH_QUICK"):     # (QUICK: developer A/B runs only)
        if prev_affinity:
            os.sched_setaffinity(0, prev_affinity)                 # the CPU baseline may use every host core
        v, info = cpu_reference_throughput(12.0, 16)
        cpu = {"value": v, "unit": "images/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]}

    if rank == 0:
        line = {"metric": METRIC if SIDE == 352 else "images/sec %dx%d fwd+decode+NMS" % (SIDE, SIDE), "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": "batch=%d %dx%d inference (backbone+FPN+head+decode+NMS) per GPU, random weights, "
                                       "NMS conf 0.001 iou 0.4" % (BATCH, SIDE, SIDE), "global_batch": world * BATCH,
                           "parallelism": "replicas x%d, no collective" % world,
                           "input": "uint8 NCHW resident in HBM, /255 fused into the stem (utils/utils.py:368)" if u8 else "fp32 NCHW resident in HBM",
                           "l2": "inputs (%d x %d MB per step, alternated) exceed the 126 MB L2; activations stream through it"
                                 % (len(xs_dev), BATCH * 3 * SIDE * SIDE * (1 if u8 else 4) // 1000000),
                           "host": host_binding or "no CPU binding (PCI topology not exposed)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * (plan.forward_launches + 1),
                "kept_boxes_per_step": kept, "parity_checked": parity is not None, "parity": parity, "roofline": roof, "cpu_baseline": cpu, "stages": stages}
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
def run_train(args, rank, world, local_rank):
    """BASELINE configs[2]: train.py loop on synthetic boxes, batch 64 per GPU (512 on 8), forward (batch-statistics BN) ->
    DetectorLoss -> backward -> ONE NCCL all-reduce of the flat 243 095-float gradient bucket -> SGD.  Weak scaling."""
    import yfv2  # noqa: F401
    import synth
    import model.detector as det
    import utils.loss as ul
    import train_ddp
    TB = 64
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    bind_to_gpu_node(local_rank)                                         # pinned input batches next to the GPU
    torch.manual_seed(2)                                                 # same initial weights on every rank
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):
        m = det.Detector(CLASSES, ANCHORS, True).to(dev).train()
    bucket = train_ddp.FlatGradBucket(m.parameters())
    opt = train_ddp.make_optimizer(m, 1e-3)
    c = cfg()
    g = torch.Generator().manual_seed(2 + rank)
    x = torch.rand(TB, 3, SIDE, SIDE, generator=g).to(dev)               # the rank's shard of the 512-image batch
    targets = synth.make_targets(2 + rank, TB).to(dev)                   # ~7 boxes per image (SURVEY 8d config[2])
    xh = (torch.rand(TB, 3, SIDE, SIDE, generator=g) * 255).to(torch.uint8).pin_memory()
    th = synth.make_targets(20 + rank, TB).pin_memory()
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def step():
        return train_ddp.train_step(m, bucket, opt, x, targets, c, ul.compute_loss)

    def e2e_step():
        xi = xh.to(dev, non_blocking=True).float() / 255.0               # train.py:101
        ti = th.to(dev, non_blocking=True)
        losses = train_ddp.train_step(m, bucket, opt, xi, ti, c, ul.compute_loss)
        return float(losses[3].detach())                                          # the loss read the reference's progress bar does every iteration

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        losses = step()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t.item())
    # the collective alone (device time, max over ranks)
    ar = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(stream)
        bucket.allreduce_mean()
        b.record(stream)
        b.synchronize()
        ar.append(a.elapsed_time(b) * 1e3)
    ar_us = torch.tensor([sorted(ar)[len(ar) // 2]], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(ar_us, op=torch.distributed.ReduceOp.MAX)
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(args.steps):
        last = e2e_step()
    s1.record(stream)
    barrier()
    t2 = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t2, op=torch.distributed.ReduceOp.MAX)
    if rank == 0:
        line = {"metric": "training images/sec 352x352 fwd+loss+bwd+allreduce+SGD", "mode": "train", "value": world * TB * args.steps / (ms / 1e3),
                "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "train.py loop, batch 64 per GPU (global %d) @352x352, synthetic boxes (1..13 per image), DetectorLoss "
                                       "backward, one NCCL all-reduce of the flat gradient bucket, SGD(momentum 0.949, wd 5e-4); default PyTorch init "
                                       "(the pretrained backbone.pth is not on the GPU box)" % (world * TB),
                           "global_batch": world * TB, "parallelism": "dp%d" % world},
                "clocks": clocks, "loss": float(losses[3].detach()),
                "allreduce": {"us": float(ar_us.item()), "bytes": bucket.flat.numel() * 4, "comm_nranks": world,
                              "collectives_per_step": 1 if world > 1 else 0},
                "e2e": {"value": world * TB * args.steps / (float(t2.item()) / 1e3), "unit": "images/s",
                        "h2d_bytes_per_step": xh.numel() + th.numel() * 4, "d2h_bytes_per_step": 4,
                        "api": "train_ddp.train_step from pinned host uint8 images + targets, loss read back every step", "last_loss": last}}
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--side", type=int, default=352, help="input height = width (640: BASELINE configs[3], 256 images per GPU)")
    ap.add_argument("--batch", type=int, default=256, help="images per GPU")
    ap.add_argument("--input", default="u8", choices=["u8", "f32"], help="dtype of the HBM-resident input batch of the device-timed step")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"], help="infer: BASELINE configs[1] (default); train: configs[2]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (head tensors, detections, counts; rank 0) as DIR/<name>.npy. "
                         "Inputs and weights are seeded, so the same arguments give the same inputs on every run and build")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the inference workload of --impl ours")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    globals().update(SIDE=args.side, BATCH=args.batch)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); use --impl reference for the CPU arm")
    if world > 1:
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.mode == "train":
            run_train(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

"""ctypes binding of libyfv2.so (include/yfv2.h) plus the small amount of host bookkeeping the Python
mirror modules share: plan cache, weight packing, output allocation.  PyTorch is used for device
memory and streams only; every device computation is a kernel inside libyfv2.so.

There is NO CPU fallback: if the library is missing or the tensors are not on a CUDA device the calls
raise.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libyfv2.so")
_lib = None
_lock = threading.Lock()

MAX_DET = 300          # reference utils/utils.py:242
MAX_WH = 4096.0        # reference utils/utils.py:241

_c_float_p = ctypes.POINTER(ctypes.c_float)
_c_void_pp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); must list every prototype of include/yfv2.h (tests check this)
PROTOTYPES = {
    "yfv2_abi_version": (ctypes.c_int, []),
    "yfv2_last_error": (ctypes.c_char_p, []),
    "yfv2_plan_create": (ctypes.c_int, [_c_void_pp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "yfv2_plan_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "yfv2_plan_workspace_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t)]),
    "yfv2_plan_invalidate_workspace": (ctypes.c_int, [ctypes.c_void_p]),
    "yfv2_plan_packed_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t)]),
    "yfv2_plan_forward_launches": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]),
    "yfv2_pack_weights": (ctypes.c_int, [ctypes.c_void_p, _c_void_pp, _c_void_pp, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, _c_void_pp, ctypes.c_void_p,
                                    ctypes.c_void_p]),
    "yfv2_forward_u8": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, _c_void_pp, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    "yfv2_decode": (ctypes.c_int, [_c_void_pp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                   ctypes.POINTER(ctypes.c_double), ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_export_heads": (ctypes.c_int, [_c_void_pp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_nms_workspace_bytes": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_size_t)]),
    "yfv2_nms": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_double,
                                ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p,
                                ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_decode_nms": (ctypes.c_int, [_c_void_pp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_double), ctypes.c_float, ctypes.c_double, ctypes.c_void_p,
                                       ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_batch_statistics": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_aug_contrast_brightness": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p]),
    "yfv2_resize_u8": (ctypes.c_int, [_c_void_pp, ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_detect_u8_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.POINTER(ctypes.c_double), ctypes.c_float, ctypes.c_double, ctypes.c_int,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_detect_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int]),
    "yfv2_loss_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 6 + [ctypes.POINTER(ctypes.c_size_t)]),
    "yfv2_compute_loss": (ctypes.c_int, [_c_void_pp, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.c_void_p, _c_void_pp,
                                         ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_loss_read_targets": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p, ctypes.c_void_p,
                                              ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_op_conv1x1_fwd": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_conv1x1_bwd": (ctypes.c_int, [ctypes.c_void_p] * 6 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_dwconv_fwd": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_void_p]),
    "yfv2_op_dwconv_bwd": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int] * 6 + [ctypes.c_void_p]),
    "yfv2_op_stem_fwd": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_stem_wgrad": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_bn_train_fwd": (ctypes.c_int, [ctypes.c_void_p] * 9 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_bn_train_bwd": (ctypes.c_int, [ctypes.c_void_p] * 10 + [ctypes.c_int] * 4 + [ctypes.c_void_p]),
    "yfv2_op_maxpool_fwd": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3 + [ctypes.c_void_p]),
    "yfv2_op_maxpool_bwd": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3 + [ctypes.c_void_p]),
    "yfv2_op_upsample2_fwd": (ctypes.c_int, [ctypes.c_void_p] * 2 + [ctypes.c_int] * 3 + [ctypes.c_void_p]),
    "yfv2_op_upsample2_bwd": (ctypes.c_int, [ctypes.c_void_p] * 2 + [ctypes.c_int] * 3 + [ctypes.c_void_p]),
    "yfv2_trainer_create": (ctypes.c_int, [_c_void_pp] + [ctypes.c_int] * 6),
    "yfv2_trainer_destroy": (None, [ctypes.c_void_p]),
    "yfv2_trainer_workspace_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t)]),
    "yfv2_trainer_grad_floats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_longlong)]),
    "yfv2_trainer_param_offset": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong)]),
    "yfv2_train_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, _c_void_pp, _c_void_pp, _c_void_pp, ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_train_backward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, _c_void_pp, _c_void_pp, _c_void_pp, ctypes.c_void_p, ctypes.c_int,
                                           ctypes.c_void_p, ctypes.c_void_p]),
    "yfv2_plan_stage_name": (ctypes.c_char_p, [ctypes.c_void_p, ctypes.c_int]),
    "yfv2_plan_stage_group": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "yfv2_forward_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, _c_void_pp,
                                          ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "yfv2_debug_pw_tc": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "yfv2_debug_gather": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                         ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]),
    "yfv2_debug_nms_profile": (ctypes.c_int, [ctypes.c_void_p]),
    "yfv2_debug_head_lanemap": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_longlong,
                                               ctypes.POINTER(ctypes.c_uint)]),
    "yfv2_ncnn_post": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_float), ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                      ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
}


def lib():
    """Loads libyfv2.so (once).  Raises if it has not been built — there is no fallback path."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(_LIB_PATH):
                    raise RuntimeError("libyfv2.so is missing (%s): build it with "
                                       "`python yolo-fastestv2_b200/build.py` or __graft_entry__.build()" % _LIB_PATH)
                L = ctypes.CDLL(_LIB_PATH)
                for name, (res, args) in PROTOTYPES.items():
                    fn = getattr(L, name)
                    fn.restype, fn.argtypes = res, args
                _lib = L
    return _lib


class Yfv2Error(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        raise Yfv2Error("%s failed (%d): %s" % (what, rc, lib().yfv2_last_error().decode("utf-8", "replace")))


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr_array(tensors):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise Yfv2Error("%s must be a CUDA tensor: this implementation has no CPU path" % name)


class Trainer:
    """One yfv2_trainer (the native train-mode forward + backward of the whole network) with its workspace.  The workspace keeps
    ONE batch's activations: backward() must follow the forward() of the same batch."""

    def __init__(self, device, N, H, W, A, C):
        L = lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise Yfv2Error("trainers exist on CUDA devices only")
        self.N, self.H, self.W, self.A, self.C = N, H, W, A, C
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _check(L.yfv2_trainer_create(ctypes.byref(self._h), self.device.index or 0, N, H, W, A, C), "trainer_create")
        nb = ctypes.c_size_t()
        _check(L.yfv2_trainer_workspace_bytes(self._h, ctypes.byref(nb)), "trainer_workspace_bytes")
        self.workspace = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
        n = ctypes.c_longlong()
        _check(L.yfv2_trainer_grad_floats(self._h, ctypes.byref(n)), "trainer_grad_floats")
        self.grad_floats = n.value
        self.param_offsets = []
        off, num = ctypes.c_longlong(), ctypes.c_longlong()
        for i in range(225):
            _check(L.yfv2_trainer_param_offset(self._h, i, ctypes.byref(off), ctypes.byref(num)), "trainer_param_offset")
            self.param_offsets.append((off.value, num.value))
        self.generation = 0                  # bumped by every forward: a backward must see the generation of its own forward
        # persistent buffers: the C side replays its two programs as CUDA graphs while every pointer stays the same
        self.x_static = torch.empty((N, 3, H, W), dtype=torch.float32, device=self.device)
        self.preds_static = self.alloc_preds()
        self.dpreds_static = [torch.empty_like(p) for p in self.preds_static]
        self.flat_static = torch.empty(self.grad_floats, dtype=torch.float32, device=self.device)

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                lib().yfv2_trainer_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass

    def alloc_preds(self):
        out = []
        for s in (16, 32):
            h, w = self.H // s, self.W // s
            for ch in (4 * self.A, self.A, self.C):
                out.append(torch.empty((self.N, ch, h, w), dtype=torch.float32, device=self.device))
        return out

    @staticmethod
    def _check_weights(params, bn_running):
        if len(params) != 225 or len(bn_running) != 146:
            raise Yfv2Error("trainer: expected 225 parameters and 146 BN buffers, got %d / %d" % (len(params), len(bn_running)))
        for t in list(params) + list(bn_running):
            _require_cuda(t, "weight")
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise Yfv2Error("trainer: weights must be contiguous float32")

    def forward(self, x, params, bn_running):
        self._check_weights(params, bn_running)
        _require_cuda(x, "x")
        if tuple(x.shape) != (self.N, 3, self.H, self.W) or x.dtype != torch.float32 or not x.is_contiguous():
            raise Yfv2Error("trainer: expected a contiguous float32 input of shape %s" % ((self.N, 3, self.H, self.W),))
        self.x_static.copy_(x)                               # (the graph reads the batch from a fixed address)
        preds = self.preds_static
        with torch.cuda.device(self.device):
            _check(lib().yfv2_train_forward(self._h, ctypes.c_void_p(self.x_static.data_ptr()), _ptr_array(params), _ptr_array(bn_running),
                                            _ptr_array(preds), ctypes.c_void_p(self.workspace.data_ptr()), _stream(self.device)),
                   "train_forward")
        self.generation += 1
        return [p.detach() for p in preds]                   # aliases of the trainer's head buffers (overwritten by the next forward)

    def backward(self, params, dpreds, grads_flat, accumulate):
        """Backward of the last forward().  grads_flat None: the trainer's own flat buffer (overwritten) is used and returned."""
        if grads_flat is None:
            grads_flat, accumulate = self.flat_static, False
        if grads_flat.numel() != self.grad_floats or grads_flat.dtype != torch.float32 or not grads_flat.is_contiguous():
            raise Yfv2Error("trainer: grads_flat must be a contiguous float32 buffer of %d elements" % self.grad_floats)
        torch._foreach_copy_(self.dpreds_static, [d if d.is_contiguous() else d.contiguous() for d in dpreds])
        with torch.cuda.device(self.device):
            _check(lib().yfv2_train_backward(self._h, ctypes.c_void_p(self.x_static.data_ptr()), _ptr_array(params),
                                             _ptr_array(self.preds_static), _ptr_array(self.dpreds_static),
                                             ctypes.c_void_p(grads_flat.data_ptr()), int(bool(accumulate)),
                                             ctypes.c_void_p(self.workspace.data_ptr()), _stream(self.device)), "train_backward")
        return grads_flat


def anchors_array(cfg):
    a = [float(v) for v in cfg["anchors"]]
    return (ctypes.c_double * len(a))(*a)


class Plan:
    """One yfv2_plan with its workspace and packed-weight buffer (owned here as torch tensors)."""

    def __init__(self, device, N, H, W, A, C, training=False, detect_max_det=0):
        L = lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise Yfv2Error("plans exist on CUDA devices only")
        self.N, self.H, self.W, self.A, self.C = N, H, W, A, C
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _check(L.yfv2_plan_create(ctypes.byref(self._h), self.device.index or 0, N, H, W, A, C, int(training)), "plan_create")
        nb = ctypes.c_size_t()
        _check(L.yfv2_plan_workspace_bytes(self._h, ctypes.byref(nb)), "workspace_bytes")
        ws_bytes = nb.value
        if detect_max_det:
            ws_bytes = max(ws_bytes, L.yfv2_detect_workspace_bytes(self._h, detect_max_det))
        self.workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        _check(L.yfv2_plan_packed_bytes(self._h, ctypes.byref(nb)), "packed_bytes")
        self.packed = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
        n = ctypes.c_int()
        _check(L.yfv2_plan_forward_launches(self._h, ctypes.byref(n)), "forward_launches")
        self.forward_launches = n.value
        self.stage_names = []                 # fused stages; stages sharing a stage_groups value are one kernel launch
        while True:
            nm = L.yfv2_plan_stage_name(self._h, len(self.stage_names))
            if nm is None:
                break
            self.stage_names.append(nm.decode())
        self.stage_groups = [L.yfv2_plan_stage_group(self._h, i) for i in range(len(self.stage_names))]
        self.packed_version = None

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                lib().yfv2_plan_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass

    def pack(self, params, bn_running):
        """params: 225 fp32 CUDA tensors in Detector.parameters() order; bn_running: 146 (mean, var, ...)."""
        if len(params) != 225 or len(bn_running) != 146:
            raise Yfv2Error("pack: expected 225 parameters and 146 BN buffers, got %d / %d" % (len(params), len(bn_running)))
        keep = []
        for t in list(params) + list(bn_running):
            _require_cuda(t, "weight")
            if t.dtype != torch.float32:
                raise Yfv2Error("weights must be float32")
            keep.append(t.detach().contiguous())
        with torch.cuda.device(self.device):
            _check(lib().yfv2_pack_weights(self._h, _ptr_array(keep[:225]), _ptr_array(keep[225:]),
                                           ctypes.c_void_p(self.packed.data_ptr()), _stream(self.device)), "pack_weights")
        return keep   # caller may drop it after the stream has run; kept alive by stream ordering of the allocator

    def alloc_preds(self):
        N, A, C = self.N, self.A, self.C
        out = []
        for s in (16, 32):
            h, w = self.H // s, self.W // s
            for ch in (4 * A, A, C):
                out.append(torch.empty((N, ch, h, w), dtype=torch.float32, device=self.device))
        return tuple(out)

    def forward(self, x, preds=None):
        _require_cuda(x, "x")
        if tuple(x.shape) != (self.N, 3, self.H, self.W):
            raise Yfv2Error("forward: input shape %s does not match the plan (%d,3,%d,%d)" % (tuple(x.shape), self.N, self.H, self.W))
        if x.dtype not in (torch.float32, torch.uint8):
            raise Yfv2Error("forward: input must be float32 or uint8")
        x = x.contiguous()
        if preds is None:
            preds = self.alloc_preds()
        fn = lib().yfv2_forward if x.dtype == torch.float32 else lib().yfv2_forward_u8
        with torch.cuda.device(self.device):
            _check(fn(self._h, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(self.packed.data_ptr()), _ptr_array(preds),
                      ctypes.c_void_p(self.workspace.data_ptr()), _stream(self.device)), "forward")
        return preds

    def forward_range(self, x, preds, first, last):
        """Runs fused stages [first,last) only (see yfv2.h); x, preds as in forward()."""
        with torch.cuda.device(self.device):
            _check(lib().yfv2_forward_range(self._h, ctypes.c_void_p(x.data_ptr()), int(x.dtype == torch.uint8),
                                            ctypes.c_void_p(self.packed.data_ptr()), _ptr_array(preds),
                                            ctypes.c_void_p(self.workspace.data_ptr()), first, last, _stream(self.device)),
                   "forward_range")

    def debug_gather(self, which):
        """Dense NCHW copy of an intermediate tensor of the last forward (test hook, see yfv2.h)."""
        dims = (ctypes.c_int * 4)()
        _check(lib().yfv2_debug_gather(self._h, ctypes.c_void_p(self.workspace.data_ptr()), which, None, dims, None), "debug_gather")
        out = torch.empty(tuple(dims), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _check(lib().yfv2_debug_gather(self._h, ctypes.c_void_p(self.workspace.data_ptr()), which,
                                           ctypes.c_void_p(out.data_ptr()), dims, _stream(self.device)), "debug_gather")
        return out

    def detect_u8_host(self, x_host, anchors, conf_thres, iou_thres, out_host, counts_host, max_det=MAX_DET):
        """Whole step from pinned host uint8 images to pinned host detections (asynchronous)."""
        with torch.cuda.device(self.device):
            _check(lib().yfv2_detect_u8_host(self._h, ctypes.c_void_p(x_host.data_ptr()), ctypes.c_void_p(self.packed.data_ptr()),
                                             anchors, ctypes.c_float(conf_thres), ctypes.c_double(iou_thres), max_det,
                                             ctypes.c_void_p(out_host.data_ptr()), ctypes.c_void_p(counts_host.data_ptr()),
                                             ctypes.c_void_p(self.workspace.data_ptr()), _stream(self.device)), "detect_u8_host")


def decode(preds, cfg):
    """handel_preds on the device: returns [N, M, 5+C] fp32 CUDA tensor."""
    for p in preds:
        _require_cuda(p, "preds")
    preds = [p.detach().contiguous().float() for p in preds]
    N, A4, h, w = preds[0].shape
    A, C = preds[1].shape[1], preds[2].shape[1]
    if len(preds) != 6 or A4 != 4 * A:
        raise Yfv2Error("decode: expected the 6-tuple (reg,obj,cls) x 2 levels")
    H, W = h * 16, w * 16
    if cfg is not None and (int(cfg["height"]) != H or int(cfg["width"]) != W):
        raise Yfv2Error("decode: head tensors are %dx%d/16 but cfg says %sx%s" % (H, W, cfg["height"], cfg["width"]))
    M = (h * w + preds[3].shape[2] * preds[3].shape[3]) * A
    out = torch.empty((N, M, 5 + C), dtype=torch.float32, device=preds[0].device)
    with torch.cuda.device(out.device):
        _check(lib().yfv2_decode(_ptr_array(preds), N, H, W, A, C, anchors_array(cfg), ctypes.c_void_p(out.data_ptr()),
                                 _stream(out.device)), "decode")
    return out


def _filter_tensor(classes, device):
    if classes is None:
        return None, 0
    classes = list(classes)
    if not classes:
        classes = [-1]      # the reference keeps rows whose class is IN the list (utils/utils.py:266-268): an empty list keeps nothing
    t = torch.as_tensor(classes, dtype=torch.int32, device=device)
    return t, t.numel()


def nms(dets, conf_thres=0.3, iou_thres=0.45, classes=None, max_det=MAX_DET, want_idx=True):
    """Device NMS.  Returns (out [N,max_det,6], counts [N] int32, kept_idx [N,max_det] int32 or None)."""
    _require_cuda(dets, "dets")
    dets = dets.detach().contiguous().float()
    N, M, D = dets.shape
    out = torch.empty((N, max_det, 6), dtype=torch.float32, device=dets.device)
    counts = torch.empty((N,), dtype=torch.int32, device=dets.device)
    idx = torch.empty((N, max_det), dtype=torch.int32, device=dets.device) if want_idx else None
    filt, nf = _filter_tensor(classes, dets.device)
    with torch.cuda.device(dets.device):
        _check(lib().yfv2_nms(ctypes.c_void_p(dets.data_ptr()), N, M, D - 5, ctypes.c_float(conf_thres), ctypes.c_double(iou_thres),
                              ctypes.c_void_p(filt.data_ptr()) if nf else None, nf, max_det, ctypes.c_float(MAX_WH),
                              ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(counts.data_ptr()),
                              ctypes.c_void_p(idx.data_ptr()) if want_idx else None, None, _stream(dets.device)), "nms")
    return out, counts, idx


def decode_nms(preds, cfg, conf_thres=0.3, iou_thres=0.45, classes=None, max_det=MAX_DET, want_idx=False):
    """Fused handel_preds + non_max_suppression on the device (no [N,M,5+C] tensor)."""
    for p in preds:
        _require_cuda(p, "preds")
    preds = [p.detach().contiguous().float() for p in preds]
    N, _, h, w = preds[0].shape
    A, C = preds[1].shape[1], preds[2].shape[1]
    H, W = h * 16, w * 16
    dev = preds[0].device
    out = torch.empty((N, max_det, 6), dtype=torch.float32, device=dev)
    counts = torch.empty((N,), dtype=torch.int32, device=dev)
    idx = torch.empty((N, max_det), dtype=torch.int32, device=dev) if want_idx else None
    filt, nf = _filter_tensor(classes, dev)
    with torch.cuda.device(dev):
        _check(lib().yfv2_decode_nms(_ptr_array(preds), N, H, W, A, C, anchors_array(cfg), ctypes.c_float(conf_thres),
                                     ctypes.c_double(iou_thres), ctypes.c_void_p(filt.data_ptr()) if nf else None, nf, max_det,
                                     ctypes.c_float(MAX_WH), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(counts.data_ptr()),
                                     ctypes.c_void_p(idx.data_ptr()) if want_idx else None, None, _stream(dev)), "decode_nms")
    return out, counts, idx


def batch_statistics(out, counts, targets, iou_threshold):
    """True-positive flags [N,max_det] (float 0/1) of NMS output rows against pixel-xyxy targets [nt,6] (device)."""
    _require_cuda(out, "out")
    N, max_det, _ = out.shape
    targets = targets.detach().to(out.device).float().contiguous().reshape(-1, 6)
    tp = torch.empty((N, max_det), dtype=torch.float32, device=out.device)
    with torch.cuda.device(out.device):
        _check(lib().yfv2_batch_statistics(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(counts.data_ptr()), N, max_det,
                                           ctypes.c_void_p(targets.data_ptr()) if targets.numel() else None, targets.shape[0],
                                           ctypes.c_float(iou_threshold), ctypes.c_void_p(tp.data_ptr()), _stream(out.device)),
               "batch_statistics")
    return tp


def contrast_and_brightness(imgs, alpha, beta, out=None):
    """utils.datasets.contrast_and_brightness (cv2.addWeighted on uint8) for a batch on the device: imgs uint8 [N, ...],
    alpha / beta float32 [N] (one pair per image).  Returns a new uint8 tensor (or writes `out`, which may be `imgs`)."""
    _require_cuda(imgs, "imgs")
    if imgs.dtype != torch.uint8:
        raise TypeError("contrast_and_brightness expects uint8 images (the reference augments before the /255)")
    imgs = imgs.contiguous()
    N = imgs.shape[0]
    alpha = torch.as_tensor(alpha, dtype=torch.float32).to(imgs.device).contiguous().reshape(-1)
    beta = torch.as_tensor(beta, dtype=torch.float32).to(imgs.device).contiguous().reshape(-1)
    if alpha.numel() != N or beta.numel() != N:
        raise ValueError("one (alpha, beta) pair per image")
    if out is None:
        out = torch.empty_like(imgs)
    with torch.cuda.device(imgs.device):
        _check(lib().yfv2_aug_contrast_brightness(ctypes.c_void_p(imgs.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                  ctypes.c_void_p(alpha.data_ptr()), ctypes.c_void_p(beta.data_ptr()), N,
                                                  imgs.numel() // N, _stream(imgs.device)), "aug_contrast_brightness")
    return out


def resize_u8(images, height, width, out=None):
    """cv2.resize(img, (width, height), interpolation=cv2.INTER_LINEAR) + transpose(2,0,1) for a batch on the device
    (utils/datasets.py:106-111, test.py:34-37): images is a list of CUDA uint8 [h,w,3] tensors of any sizes (rows contiguous; views
    at any byte offset are fine).  Returns CUDA uint8 [N,3,height,width] (or writes `out`)."""
    images = list(images)
    if not images:
        raise ValueError("resize_u8: no images")
    for im in images:
        _require_cuda(im, "images")
        if im.dtype != torch.uint8 or im.dim() != 3 or im.shape[2] != 3:
            raise Yfv2Error("resize_u8: images must be uint8 [h, w, 3], got %s %s" % (im.dtype, tuple(im.shape)))
        if im.stride() != (3 * im.shape[1], 3, 1):
            raise Yfv2Error("resize_u8: image rows must be contiguous")
    dev = images[0].device
    N = len(images)
    if out is None:
        out = torch.empty((N, 3, height, width), dtype=torch.uint8, device=dev)
    elif tuple(out.shape) != (N, 3, height, width) or out.dtype != torch.uint8 or not out.is_contiguous() or out.device != dev:
        raise Yfv2Error("resize_u8: out must be a contiguous uint8 [%d,3,%d,%d] tensor on %s" % (N, height, width, dev))
    hw = (ctypes.c_int * (2 * N))(*[int(v) for im in images for v in im.shape[:2]])
    with torch.cuda.device(dev):
        _check(lib().yfv2_resize_u8(_ptr_array(images), hw, N, height, width, ctypes.c_void_p(out.data_ptr()), _stream(dev)),
               "resize_u8")
    return out


def debug_pw_tc(x, w):
    """out[n][p] = sum_k w[n][k] * x[k][p] on the tcgen05 3xTF32 engine (test hook)."""
    _require_cuda(x, "x"); _require_cuda(w, "w")
    K, P = x.shape
    N = w.shape[0]
    out = torch.empty((N, P), dtype=torch.float32, device=x.device)
    ws = torch.empty((2 * ((N + 15) // 16 * 16) * ((K + 7) // 8 * 8),), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _check(lib().yfv2_debug_pw_tc(ctypes.c_void_p(x.contiguous().data_ptr()), ctypes.c_void_p(w.contiguous().data_ptr()),
                                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ws.data_ptr()), K, N, P, _stream(x.device)),
               "debug_pw_tc")
    return out


def compute_loss(preds, targets, cfg, want_grads=True, return_workspace=False):
    """utils.loss.compute_loss on the device.  Returns (losses[4] CUDA tensor, dpreds 6-tuple or None[, workspace])."""
    for p in preds:
        _require_cuda(p, "preds")
    preds = [p.detach().contiguous().float() for p in preds]
    N, A4, h, w = preds[0].shape
    A, C = preds[1].shape[1], preds[2].shape[1]
    H, W = h * 16, w * 16
    dev = preds[0].device
    targets = targets.detach().to(dev).float().contiguous().reshape(-1, 6)
    nt = targets.shape[0]
    nb = ctypes.c_size_t()
    _check(lib().yfv2_loss_workspace_bytes(N, H, W, A, C, nt, ctypes.byref(nb)), "loss_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    losses = torch.empty(4, dtype=torch.float32, device=dev)
    dpreds = [torch.empty_like(p) for p in preds] if want_grads else None
    with torch.cuda.device(dev):
        _check(lib().yfv2_compute_loss(_ptr_array(preds), ctypes.c_void_p(targets.data_ptr()) if nt else None, nt, N, H, W, A, C,
                                       anchors_array(cfg), ctypes.c_void_p(losses.data_ptr()),
                                       _ptr_array(dpreds) if want_grads else None, ctypes.c_void_p(ws.data_ptr()), _stream(dev)),
               "compute_loss")
    out = (losses, tuple(dpreds) if want_grads else None)
    return out + ((ws, (N, H, W, A, nt)),) if return_workspace else out


def read_targets(ws_info, level):
    """Matched rows of one level after compute_loss(..., return_workspace=True): (idx[4,m], tbox[m,4], anch[m,2], tcls[m])."""
    ws, (N, H, W, A, nt) = ws_info
    cap = 5 * A * max(nt, 1)
    dev = ws.device
    idx = torch.zeros((4, cap), dtype=torch.int32, device=dev)
    tbox = torch.zeros((cap, 4), dtype=torch.float32, device=dev)
    anch = torch.zeros((cap, 2), dtype=torch.float64, device=dev)
    tcls = torch.zeros((cap,), dtype=torch.int32, device=dev)
    cnt = ctypes.c_int()
    with torch.cuda.device(dev):
        _check(lib().yfv2_loss_read_targets(ctypes.c_void_p(ws.data_ptr()), level, N, H, W, A, nt, ctypes.byref(cnt),
                                            ctypes.c_void_p(idx.data_ptr()), ctypes.c_void_p(tbox.data_ptr()),
                                            ctypes.c_void_p(anch.data_ptr()), ctypes.c_void_p(tcls.data_ptr()), _stream(dev)),
               "loss_read_targets")
    m = cnt.value
    return idx[:, :m], tbox[:m], anch[:m], tcls[:m]


def op(name, tensors_and_ints, device):
    """Calls yfv2_op_<name>: tensors become data pointers (None -> NULL), ints pass through, the stream is appended."""
    args = []
    for a in tensors_and_ints:
        if a is None:
            args.append(None)
        elif isinstance(a, torch.Tensor):
            args.append(ctypes.c_void_p(a.data_ptr()))
        else:
            args.append(int(a))
    with torch.cuda.device(device):
        _check(getattr(lib(), "yfv2_op_" + name)(*args, _stream(device)), "op_" + name)


def export_heads(preds):
    """Detector(..., export_onnx=True) output: two channel-last [N,h,w,5A+C] tensors (sigmoid / sigmoid / softmax)."""
    preds = [p.detach().contiguous().float() for p in preds]
    N, _, h, w = preds[0].shape
    A, C = preds[1].shape[1], preds[2].shape[1]
    dev = preds[0].device
    o2 = torch.empty((N, h, w, 5 * A + C), dtype=torch.float32, device=dev)
    o3 = torch.empty((N, preds[3].shape[2], preds[3].shape[3], 5 * A + C), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(lib().yfv2_export_heads(_ptr_array(preds), N, h * 16, w * 16, A, C, ctypes.c_void_p(o2.data_ptr()),
                                       ctypes.c_void_p(o3.data_ptr()), _stream(dev)), "export_heads")
    return o2, o3


NCNN_ANCHORS = (12.64, 19.39, 37.88, 51.48, 55.71, 138.31, 126.91, 78.23, 131.57, 214.55, 279.92, 258.87)   # sample/ncnn/src/yolo-fastestv2.cpp:34-35


def ncnn_post(out2, out3, anchor_num, thresh=0.3, nms_thresh=0.25, src_size=None, anchors=NCNN_ANCHORS, max_out=None):
    """The deploy post-process of the reference's ncnn sample (yoloFastestv2::detection after the forward: predHandle + nmsHandle,
    sample/ncnn/src/yolo-fastestv2.cpp:78-183) on the export_onnx tensors `out2` [N,h,w,5A+C], `out3` (export_heads above).
    src_size = (cols, rows) of the source image (default: the network input size, scale 1).  Returns a list of N tuples
    (boxes int32 [n,4], scores float32 [n], cates int32 [n]) on the CPU, descending score, like the sample's dstBoxes."""
    if not (out2.is_cuda and out3.is_cuda):
        raise RuntimeError("yfv2: ncnn_post needs CUDA tensors (there is no CPU fallback)")
    out2 = out2.detach().contiguous().float(); out3 = out3.detach().contiguous().float()
    N, h, w, ch = out2.shape
    A = int(anchor_num)
    C = ch - 5 * A
    H, W = h * 16, w * 16
    M = A * (h * w + out3.shape[1] * out3.shape[2])
    max_out = M if max_out is None else int(max_out)
    sw, sh = (W, H) if src_size is None else src_size
    import numpy as np
    scale_w = float(np.float32(sw) / np.float32(W)); scale_h = float(np.float32(sh) / np.float32(H))        # :189-190, float division
    dev = out2.device
    boxes = torch.empty((N, max_out, 4), dtype=torch.int32, device=dev)
    scores = torch.empty((N, max_out), dtype=torch.float32, device=dev)
    cates = torch.empty((N, max_out), dtype=torch.int32, device=dev)
    counts = torch.empty((N,), dtype=torch.int32, device=dev)
    if len(anchors) < 4 * A:
        raise Yfv2Error("ncnn_post: %d anchor values given, 2 levels x %d anchors x (w, h) needed" % (len(anchors), A))
    if C <= 0:
        raise Yfv2Error("ncnn_post: tensors with %d channels cannot hold %d anchors" % (ch, A))
    anc = (ctypes.c_float * (4 * A))(*[float(a) for a in anchors][:4 * A])
    with torch.cuda.device(dev):
        _check(lib().yfv2_ncnn_post(ctypes.c_void_p(out2.data_ptr()), ctypes.c_void_p(out3.data_ptr()), N, H, W, A, C, anc,
                                    ctypes.c_float(thresh), ctypes.c_float(nms_thresh), ctypes.c_float(scale_w), ctypes.c_float(scale_h),
                                    max_out, ctypes.c_void_p(boxes.data_ptr()), ctypes.c_void_p(scores.data_ptr()),
                                    ctypes.c_void_p(cates.data_ptr()), ctypes.c_void_p(counts.data_ptr()), _stream(dev)), "ncnn_post")
    cnt = counts.cpu().tolist()
    b, s, c = boxes.cpu(), scores.cpu(), cates.cpu()
    return [(b[i, :min(cnt[i], max_out)].numpy(), s[i, :min(cnt[i], max_out)].numpy(), c[i, :min(cnt[i], max_out)].numpy()) for i in range(N)]

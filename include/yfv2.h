/*
 * yfv2.h — C ABI of libyfv2.so, the B200 (sm_100a) implementation of the Yolo-FastestV2 hot path.
 *
 * The reference (dog-qiuqiu/Yolo-FastestV2 @ ac2a5e3) has no FFI of its own: its boundary is the
 * Python import surface (SURVEY.md 8b).  Each entry point below replaces one reference function; the
 * Python mirror modules under yolo-fastestv2_b200/{model,utils}/ call these through ctypes and give
 * the result the reference's return types.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  Every function returns 0 on success or a negative
 *     YFV2_E* code; yfv2_last_error() returns a thread-local message for the last failure.
 *   - All `float*` / `void*` tensor arguments are DEVICE pointers unless the name ends in `_host`.
 *   - The caller owns every buffer (inputs, outputs, packed weights, workspace).  The library never
 *     allocates or frees device memory; the only state is the opaque host-side yfv2_plan.
 *   - `stream` is a cudaStream_t passed as void* (Python: torch.cuda.current_stream().cuda_stream).
 *     All launches are asynchronous on it; nothing here synchronises the device, except the
 *     *_host convenience calls which say so.
 *   - No C++ exception crosses the ABI.  There is no CPU fallback: without a CUDA device every
 *     compute entry point returns YFV2_ECUDA.
 */
#ifndef YFV2_H_
#define YFV2_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YFV2_OK            0
#define YFV2_EINVAL       -1   /* bad argument (null pointer, unsupported shape) */
#define YFV2_ECUDA        -2   /* a CUDA runtime call or launch failed */
#define YFV2_EUNSUPPORTED -3   /* valid request this build does not implement */
#define YFV2_ENOMEM       -4   /* host allocation failed / workspace too small */

#define YFV2_ABI_VERSION   1

#if defined(__GNUC__)
#define YFV2_API __attribute__((visibility("default")))
#else
#define YFV2_API
#endif

/* Number of float tensors yfv2_pack_weights consumes, in reference state_dict order:
 * 225 parameters (Detector.parameters(), model/detector.py:8-19) and 73 BatchNorm layers. */
#define YFV2_NUM_PARAMS    225
#define YFV2_NUM_BN         73
#define YFV2_NUM_GRADS  243095  /* 80 classes, 3 anchors */

typedef struct yfv2_plan yfv2_plan;

YFV2_API int         yfv2_abi_version(void);
YFV2_API const char* yfv2_last_error(void);

/* ---- plan -----------------------------------------------------------------------------------------
 * One plan per (device, N, H, W, A, C, training).  H and W must be multiples of 32
 * (model/backbone/shufflenetv2.py strides; utils/loss.py:78).  Replaces Detector.__init__'s shape
 * bookkeeping (model/detector.py:8-19). */
YFV2_API int yfv2_plan_create(yfv2_plan** plan, int device, int N, int H, int W, int A, int C, int training);
YFV2_API int yfv2_plan_destroy(yfv2_plan* plan);
YFV2_API int yfv2_plan_workspace_bytes(const yfv2_plan* plan, size_t* bytes);
/* The workspace is caller-owned but DEDICATED to the plan while the plan is in use: activation planes live in it inside
 * zero frames (the padding of every 3x3 / 5x5 convolution) which the first forward on a given workspace pointer writes
 * once and later forwards rely on.  If the memory was used for anything else in between, or was freed and re-allocated
 * (a caching allocator may hand back the same address), call yfv2_plan_invalidate_workspace() before the next forward. */
YFV2_API int yfv2_plan_invalidate_workspace(yfv2_plan* plan);
YFV2_API int yfv2_plan_packed_bytes(const yfv2_plan* plan, size_t* bytes);
/* number of kernels one yfv2_forward / yfv2_detect launches (for bench.py's gpu_launches) */
YFV2_API int yfv2_plan_forward_launches(const yfv2_plan* plan, int* n);

/* ---- weights ----------------------------------------------------------------------------------------
 * params:     225 device pointers, Detector.parameters() order (== state_dict order without buffers).
 * bn_running: 146 device pointers, (running_mean, running_var) for each of the 73 BatchNorm2d in
 *             state_dict order.  Eval plans fold BN into per-channel scale/shift kept next to the
 *             transposed conv weights (eps = 1e-5, nn.BatchNorm2d default used by the reference). */
YFV2_API int yfv2_pack_weights(yfv2_plan* plan, const float* const* params, const float* const* bn_running,
                      void* packed, void* stream);

/* ---- Detector.forward (model/detector.py:21-31,46-47) ------------------------------------------------
 * x: [N,3,H,W] fp32 NCHW in [0,1] (BGR).  preds: six dense NCHW tensors
 * (reg_2 [N,4A,H/16,W/16], obj_2 [N,A,..], cls_2 [N,C,..], reg_3, obj_3, cls_3 at H/32) raw logits. */
YFV2_API int yfv2_forward(yfv2_plan* plan, const float* x, const void* packed, float* const preds[6],
                 void* workspace, void* stream);
/* Same, from uint8 [N,3,H,W]: fuses the `imgs.float() / 255.0` of utils/utils.py:368, test.py:38,
 * train.py:101 into the stem kernel's load. */
YFV2_API int yfv2_forward_u8(yfv2_plan* plan, const uint8_t* x, const void* packed, float* const preds[6],
                    void* workspace, void* stream);

/* ---- handel_preds (utils/utils.py:303-358) -----------------------------------------------------------
 * anchors_host: 2*A*2 doubles (level-major, cfg["anchors"]).  out: [N, (H/16*W/16 + H/32*W/32)*A, 5+C]
 * fp32, row (y*w+x)*A+a within a level, stride-16 level first.  img_h is cfg["height"] (the reference
 * derives ONE stride from it for both axes, utils/utils.py:332). */
YFV2_API int yfv2_decode(const float* const preds[6], int N, int H, int W, int A, int C,
                const double* anchors_host, float* out, void* stream);

/* ---- export_onnx head (model/detector.py:33-44): sigmoid(reg) | sigmoid(obj) | softmax(cls), channel-last --------------
 * out2: [N, H/16, W/16, 5A+C], out3: [N, H/32, W/32, 5A+C] (what Detector(..., export_onnx=True).forward returns). */
YFV2_API int yfv2_export_heads(const float* const preds[6], int N, int H, int W, int A, int C, float* out2, float* out3,
                               void* stream);

/* ---- deploy post-process: what yoloFastestv2::detection does after the forward (sample/ncnn/src/yolo-fastestv2.cpp) --------
 * predHandle (:134-183: cls*obj first strict maximum above 0, grid decode in double, corners (c -/+ w/2)*scale truncated to
 * int) + nmsHandle (:78-110: descending score, greedy, suppressed iff IoU > nms_thresh with a kept box of the SAME class;
 * IoU on the int corners, :58-71) on the two export_onnx tensors of yfv2_export_heads.  H, W: network input size (inputHeight /
 * inputWidth); anchors_host: 2*A*2 floats (the sample's `bias`, :34-37); scale_w/h: source image size / network input size
 * (:189-190).  Outputs per image, descending score: boxes [N,max_out,4] int32 (x1,y1,x2,y2), scores [N,max_out], cates
 * [N,max_out] int32, counts [N] = number kept (rows past min(count, max_out): zeros / cate -1; the sample has no cap, so pass
 * max_out = A*(H/16*W/16 + H/32*W/32) to never truncate).  Equal scores keep push order (the sample's std::sort leaves it open). */
YFV2_API int yfv2_ncnn_post(const float* out2, const float* out3, int N, int H, int W, int A, int C, const float* anchors_host,
                            float thresh, float nms_thresh, float scale_w, float scale_h, int max_out, int* boxes, float* scores,
                            int* cates, int* counts, void* stream);

/* ---- non_max_suppression (utils/utils.py:232-296) + torchvision.ops.nms ------------------------------
 * dets: [N,M,5+C].  out: [N,max_det,6] rows (x1,y1,x2,y2,conf,cls) by descending conf; counts: [N];
 * kept_idx (optional, may be NULL): [N,max_det] row index into dets[n].  class_filter: n_filter device
 * ints or NULL.  Candidates per image are limited to YFV2_NMS_MAX_CAND (the reference's max_nms=30000
 * branch, utils/utils.py:278-280, cannot trigger below that); larger M returns YFV2_EUNSUPPORTED.
 * The reference's 1-second wall-clock abort (utils/utils.py:292-294) is not reproduced. */
#define YFV2_NMS_MAX_CAND 8192
YFV2_API int yfv2_nms_workspace_bytes(int N, int M, int C, size_t* bytes);
YFV2_API int yfv2_nms(const float* dets, int N, int M, int C, float conf_thres, double iou_thres,
             const int* class_filter, int n_filter, int max_det, float max_wh,
             float* out, int* counts, int* kept_idx, void* workspace, void* stream);

/* Fused decode + NMS straight from the six head tensors (no [N,M,5+C] round trip through HBM);
 * bit-identical to yfv2_decode followed by yfv2_nms. */
YFV2_API int yfv2_decode_nms(const float* const preds[6], int N, int H, int W, int A, int C,
                    const double* anchors_host, float conf_thres, double iou_thres,
                    const int* class_filter, int n_filter, int max_det, float max_wh,
                    float* out, int* counts, int* kept_idx, void* workspace, void* stream);

/* ---- get_batch_statistics (utils/utils.py:184-230): true-positive flags of NMS output rows ----------------
 * dets [N,max_det,6] / counts [N] as yfv2_nms writes them; targets [nt,6] rows (image, class, x1, y1, x2, y2) in
 * pixels (what evaluation() builds at utils/utils.py:372-375), nt <= 8192.  tp [N,max_det] receives 1.0 for a true
 * positive, 0.0 otherwise (rows past counts[n] are 0).  Same greedy order and the same fp32 IoU (+1 convention) as the
 * reference: bit-identical flags. */
YFV2_API int yfv2_batch_statistics(const float* dets, const int* counts, int N, int max_det, const float* targets, int nt,
                                   float iou_threshold, float* tp, void* stream);

/* ---- contrast_and_brightness (utils/datasets.py:10-16; the augmentation img_aug applies, :63-68) on the device ----
 * out = cv2.addWeighted(img, alpha[n], zeros, 1 - alpha[n], beta[n]) for uint8 images: per byte
 * saturate_cast<uint8>(cvRound(fl32(fl32(x * alpha) + beta))).  img / out: N images of bytes_per_image bytes each (any
 * layout: the operation is elementwise; in place allowed); alpha / beta: device arrays [N] (the reference draws both from
 * random.uniform(0.25, 1.75) per image on the host).  Bit-identical to OpenCV 4.x. */
YFV2_API int yfv2_aug_contrast_brightness(const uint8_t* img, uint8_t* out, const float* alpha, const float* beta, int N,
                                          long long bytes_per_image, void* stream);

/* ---- cv2.resize(img, (W, H), interpolation=cv2.INTER_LINEAR) + transpose(2,0,1) on the device -------------------------------
 * The first step of every input path of the reference: utils/datasets.py:106-111 (TensorDataset.__getitem__, behind train.py
 * and evaluation()) and test.py:34-37, both right after cv2.imread.  src: HOST array of N device pointers, one HWC uint8 image
 * each (3 channels, rows contiguous: 3*w bytes; any byte alignment); src_hw: HOST array [N][2] of (h, w).  out: device uint8
 * [N,3,H,W], the input of yfv2_forward_u8; channel order is kept.  Bit-identical to OpenCV 4.x's uint8 INTER_LINEAR (its fixed-
 * point coefficients and rounding, incl. the exact 2x / 3x downscales it routes through INTER_AREA).  Both host arrays are read
 * before the call returns (the descriptors travel in kernel parameters, 256 images per launch).  Arguments are checked before
 * any launch: null pointers, N <= 0, an empty size or `out` overlapping a source give YFV2_EINVAL, sizes above the limits
 * below YFV2_EUNSUPPORTED. */
#define YFV2_RESIZE_MAX_SRC 8192   /* source h, w */
#define YFV2_RESIZE_MAX_DST 1024   /* destination H, W */
YFV2_API int yfv2_resize_u8(const uint8_t* const* src, const int* src_hw, int N, int H, int W, uint8_t* out, void* stream);

/* ---- whole inference step with HOST buffers (the evaluation() inner loop, utils/utils.py:367-383) ----
 * x_host: pinned uint8 [N,3,H,W]; out_host: pinned [N,max_det,6]; counts_host: pinned [N].
 * Copies in, runs forward_u8 + decode_nms, copies out, all on `stream`; returns without synchronising. */
YFV2_API int yfv2_detect_u8_host(yfv2_plan* plan, const uint8_t* x_host, const void* packed,
                        const double* anchors_host, float conf_thres, double iou_thres, int max_det,
                        float* out_host, int* counts_host, void* workspace, void* stream);
YFV2_API size_t yfv2_detect_workspace_bytes(const yfv2_plan* plan, int max_det);

/* ---- compute_loss (utils/loss.py:130-208) with build_target (:53-124) and CIoU (:8-51) ---------------------------
 * preds: the six head tensors (as returned by yfv2_forward or by any other model), targets: device [nt,6] fp32 rows
 * (img_idx, cls, cx, cy, w, h) normalised; anchors_host as for yfv2_decode.  losses: device float[4] =
 * (lbox*3.2, lobj*64, lcls*32, sum) — the four values the reference returns.  dpreds (optional, may be NULL): six
 * tensors shaped like preds receiving d(loss)/d(preds) (what loss.backward() would put into the head tensors).
 * Asynchronous on `stream`; workspace from yfv2_loss_workspace_bytes. */
YFV2_API int yfv2_loss_workspace_bytes(int N, int H, int W, int A, int C, int nt, size_t* bytes);
YFV2_API int yfv2_compute_loss(const float* const preds[6], const float* targets, int nt, int N, int H, int W, int A, int C,
                               const double* anchors_host, float* losses, float* const dpreds[6], void* workspace,
                               void* stream);
/* test hook: copy out the matched rows of one pyramid level in the reference's order (offset type, anchor, target):
 * idx = device int32 [4][5*A*nt] rows (b, a, gj, gi), tbox device [.,4] fp32, anch device [.,2] fp64, tcls device int32.
 * Synchronises `stream` to return the row count. */
YFV2_API int yfv2_loss_read_targets(const void* workspace, int level, int N, int H, int W, int A, int nt, int* count_host,
                                    int* idx, float* tbox, double* anch, int* tcls, void* stream);

/* ---- training operators (train-mode forward with batch-statistics BatchNorm, and the backward of every op) --------
 * Dense NCHW fp32 device tensors; composed into the network by the Python mirror's autograd Functions
 * (yolo-fastestv2_b200/model/train_ops.py).  Reference: what autograd does for train.py:105-110.
 *   conv1x1:  y[n][m][p] = sum_k w[m][k] x[n][k][p] (+bias);  bwd outputs are optional (NULL to skip).
 *   dwconv:   depthwise ks x ks (3|5), stride 1|2, pad ks/2.   stem: dense 3x3 s2 p1 with 3 input channels.
 *   bn_train: batch statistics over (N, HW), running-stat update (momentum 0.1, unbiased var), optional fused ReLU;
 *             scratch = 2*C doubles; save_mean / save_invstd feed the backward.
 *   maxpool:  3x3 s2 p1 with argmax indices;  upsample2: nearest x2. */
YFV2_API int yfv2_op_conv1x1_fwd(const float* x, const float* w, const float* bias, float* y, int N, int K, int M, int HW, void* stream);
YFV2_API int yfv2_op_conv1x1_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* dbias, int N, int K, int M,
                                 int HW, void* stream);
YFV2_API int yfv2_op_dwconv_fwd(const float* x, const float* w, float* y, int N, int C, int H, int W, int ks, int stride, void* stream);
YFV2_API int yfv2_op_dwconv_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, int N, int C, int H, int W, int ks,
                                int stride, void* stream);
YFV2_API int yfv2_op_stem_fwd(const float* x, const float* w, float* y, int N, int M, int H, int W, void* stream);
YFV2_API int yfv2_op_stem_wgrad(const float* x, const float* dy, float* dw, int N, int M, int H, int W, void* stream);
YFV2_API int yfv2_op_bn_train_fwd(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var, float* y,
                                  float* save_mean, float* save_invstd, double* scratch, int N, int C, int HW, int relu, void* stream);
YFV2_API int yfv2_op_bn_train_bwd(const float* x, const float* y, const float* dy, const float* gamma, const float* save_mean,
                                  const float* save_invstd, float* dx, float* dgamma, float* dbeta, double* scratch, int N, int C, int HW,
                                  int relu, void* stream);
YFV2_API int yfv2_op_maxpool_fwd(const float* x, float* y, int* idx, int planes, int H, int W, void* stream);
YFV2_API int yfv2_op_maxpool_bwd(const float* dy, const int* idx, float* dx, int planes, int H, int W, void* stream);
YFV2_API int yfv2_op_upsample2_fwd(const float* x, float* y, int planes, int H, int W, void* stream);
YFV2_API int yfv2_op_upsample2_bwd(const float* dy, float* dx, int planes, int H, int W, void* stream);

/* ---- native training step: the train-mode forward and the backward of the WHOLE network as one call each ----------------
 * Replaces what nn.Module.train() + autograd do for the reference's train.py:105-110 over model/detector.py:21-31 (batch-statistics
 * BatchNorm incl. running-stat updates, ShuffleV2 shuffle / split / concat, FPN, heads, output convs).  Everything sits in a
 * caller-owned workspace laid out at create time (activations the backward needs, their gradients, scratch); no allocation per step.
 *   params[YFV2_NUM_PARAMS] / bn_running[2*YFV2_NUM_BN]: as yfv2_pack_weights (model.parameters() order; running_mean, running_var
 *     per BatchNorm layer — updated in place with momentum 0.1, num_batches_tracked is the caller's).
 *   x: fp32 [N,3,H,W].  preds[6]: the raw head tensors (written by forward; read again by backward).
 *   dpreds[6]: d(loss)/d(preds) (e.g. from yfv2_compute_loss).  grads_flat: ONE buffer of yfv2_trainer_grad_floats() floats holding
 *     every parameter's gradient at yfv2_trainer_param_offset(i) in parameter order (the bucket a data-parallel step all-reduces);
 *     accumulate != 0 adds to it (gradient accumulation over sub-batches, train.py:122-124), 0 overwrites.
 * yfv2_train_backward must follow the yfv2_train_forward of the same batch on the same workspace (and stream order). */
typedef struct yfv2_trainer yfv2_trainer;
YFV2_API int yfv2_trainer_create(yfv2_trainer** out, int device, int N, int H, int W, int A, int C);
YFV2_API void yfv2_trainer_destroy(yfv2_trainer* t);
YFV2_API int yfv2_trainer_workspace_bytes(const yfv2_trainer* t, size_t* bytes);
YFV2_API int yfv2_trainer_grad_floats(const yfv2_trainer* t, long long* n);
YFV2_API int yfv2_trainer_param_offset(const yfv2_trainer* t, int index, long long* offset, long long* numel);
YFV2_API int yfv2_train_forward(yfv2_trainer* t, const float* x, const float* const* params, float* const* bn_running,
                                float* const preds[6], void* workspace, void* stream);
YFV2_API int yfv2_train_backward(yfv2_trainer* t, const float* x, const float* const* params, float* const preds[6],
                                 const float* const dpreds[6], float* grads_flat, int accumulate, void* workspace, void* stream);

/* ---- stage-granular forward (profiling / tests) ---------------------------------------------------------
 * A forward is a list of fused stages; yfv2_plan_stage_name(i) names them ("stem", "stage2.0", ...,
 * "stage4.1/pw1", "stage4.1/dwpw", "fpn.S3", "fpn.S2", "heads2.a", ...).  yfv2_forward_range runs stages
 * [first,last) (last < 0: to the end).  Consecutive stages with the same yfv2_plan_stage_group() value are ONE
 * kernel launch when the range covers them (chained stride-1 ShuffleV2 blocks, csrc/k_blk.cu); a range that cuts
 * a group runs the covered part as its own launch, so every block output can still be tapped.
 * yfv2_plan_forward_launches() counts the launches of a whole forward.  A block's output is only intact until a
 * later stage recycles its planes. */
YFV2_API const char* yfv2_plan_stage_name(const yfv2_plan* plan, int i);
YFV2_API int yfv2_plan_stage_group(const yfv2_plan* plan, int i);    /* index of the first stage of stage i's launch; -1: bad i */
YFV2_API int yfv2_forward_range(yfv2_plan* plan, const void* x, int is_u8, const void* packed, float* const preds[6],
                                void* workspace, int first, int last, void* stream);

/* ---- test hook: dense NCHW copy of an intermediate tensor of the last forward -------------------------
 * which: 0 stem output, 1..16 ShuffleV2 block outputs in network order (logical channel order, i.e. what
 * the reference's block returns), 17 S2, 18 S3, 19..22 mid-head scratch (cls2, reg2, cls3, reg3).
 * dims4 receives [N,C,h,w]; out may be NULL to query dims only. */
YFV2_API int yfv2_debug_gather(const yfv2_plan* plan, const void* workspace, int which, float* out, int* dims4,
                               void* stream);

/* ---- test hook: one pointwise contraction on the tcgen05 engine (3xTF32), out[n][p] = sum_k w[n][k]*x[k][p] ----
 * x: [K][P], w: [N][K], out: [N][P], pack_ws: scratch of at least 2*roundup(N,16)*roundup(K,8) floats. */
YFV2_API int yfv2_debug_pw_tc(const float* x, const float* w, float* out, float* pack_ws, int K, int N, int P,
                              void* stream);

/* ---- test hook (host only, no GPU needed): the lane map the heads' pixel-pair kernel uses for an H x W map in zero frames of
 * row stride WS / plane stride PS floats, `imgs` images per work item: out[256] = image << 16 | row << 8 | pair column, or
 * 0xFFFFFFFF for an idle lane.  Every pair appears exactly once; the 16 lanes of a half-warp sit in different 8-byte banks
 * wherever the geometry allows it. */
YFV2_API int yfv2_debug_head_lanemap(int H, int W, int WS, int imgs, long long PS, unsigned int* out);

/* ---- profiling hook: yfv2_decode_nms runs an instrumented kernel while dev_buf != NULL and writes, per image, 16 int64:
 * clock64 ticks of [0] candidate generation, [1] sort, [2] staging of the first chunk, [3] chunk vs kept, [4] pairs inside the
 * chunk, [5] resolve + append, [6] unused, [7] tail; [8] chunks, [9] candidates, [10] kept.  dev_buf: N x 16 int64 on the device. */
YFV2_API int yfv2_debug_nms_profile(long long* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* YFV2_H_ */

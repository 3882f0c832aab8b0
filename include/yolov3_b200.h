/* yolov3_b200 — C ABI of the Blackwell-native (sm_100a) YOLOv3 detection hot path.
 *
 * The reference (ultralytics/yolov3, pure Python) has no FFI: its seams for this path are Python call signatures
 * (SURVEY.md §8b).  This header is the drop-in boundary a binding for those seams attaches to; each entry point cites
 * the reference interface it replaces.  Conventions:
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers owned by the caller (PyTorch);
 *   - every function returns Y3_OK (0) or a negative Y3_ERR_*; text via y3_last_error(); nothing throws;
 *   - nothing allocates device memory, nothing synchronises the stream (the only host sync is y3_model_create's
 *     one-off capability probe); all launches go to the caller's stream and are CUDA-graph capturable;
 *   - re-entrant: no global mutable state besides the last-error string (thread-local) and a mutex-guarded
 *     per-process driver-entry-point cache.  A y3_model is immutable after create.
 * Activation layout ("padded NHWC"): bf16 [n, h+2, w+2, ld] with a one-pixel all-zero halo; a tensor may be a channel
 * slice [coff, coff+c) of a wider buffer (zero-copy Concat, models/common.py:424-428).
 */
#ifndef YOLOV3_B200_H
#define YOLOV3_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Y3_OK 0
#define Y3_ERR_BAD_ARG (-1)     /* shape/alignment/enum not supported by this path */
#define Y3_ERR_CUDA (-2)        /* a CUDA runtime/driver call failed (message in y3_last_error) */
#define Y3_ERR_UNSUPPORTED (-3) /* device is not sm_100 (no fallback path exists by design) */

#define Y3_ACT_NONE 0
#define Y3_ACT_SILU 1

typedef void* y3_stream_t; /* cudaStream_t */

int y3_version(void);
/* Copies the calling thread's last error text into buf (NUL-terminated); returns its length. */
int y3_last_error(char* buf, size_t n);
/* Y3_OK iff the current CUDA device is compute capability 10.x. */
int y3_device_check(void);
/* sizeof() of the ABI structs, for bindings to verify their mirror definitions:
 * 0 y3_conv_desc, 1 y3_first_desc, 2 y3_pool_desc, 3 y3_detect_level, 4 y3_decode_desc, 5 y3_op, 6 y3_nms_params,
 * 7 y3_loss_desc. */
int64_t y3_abi_sizeof(int32_t which);
/* Programmatic dependent launch between consecutive kernels of a stream (on by default; env Y3_PDL=0 or on=0 turns it off).
 * Results are identical either way — only the launch boundaries overlap.  Returns the previous setting.  A tuning switch with
 * no counterpart in the reference. */
int y3_set_pdl(int32_t on);
/* Kernel-variant switch of y3_bn_act_bwd (non-upsample layers): 1 (default) = the cp.async shared-memory-ring kernels (three
 * work units requested ahead per thread), 0 = the register-staged ones.  Same unit order and arithmetic: results are
 * bit-identical (profiles/r02_ab_shot_kernel_variants.jsonl).  Env Y3_BN_ASYNC=0/1 sets the initial value.  Returns the
 * previous setting.  A tuning switch with no counterpart in the reference. */
int y3_set_bn_async(int32_t on);

/* ---------------------------------------------------------------------------------------------------------------
 * Conv + folded-BN + SiLU (+ residual add, + nearest-2x upsample, + concat-offset store, or fp32 head store).
 * Replaces Conv.forward_fuse (models/common.py:77-81) after BaseModel.fuse (models/yolo.py:163-172), the shortcut add
 * of Bottleneck.forward (common.py:163-165), nn.Upsample+Concat (models/yolov3.yaml:43-44,51-52) and Detect.m[i]
 * (models/yolo.py:96-98).  tcgen05 implicit GEMM; c_in % 16 == 0, c_out_pad = c_out rounded up to the tile N.
 * ksize 1|3 with stride 1, or ksize 3 with stride 2 (h, w even); pad = ksize/2.
 */
typedef struct y3_conv_desc {
  int32_t n, h, w;       /* batch, UNPADDED input height/width */
  int32_t c_in, c_out;   /* logical channels */
  int32_t ksize, stride;
  int32_t act;           /* Y3_ACT_* */
  const void* in;        /* padded NHWC bf16 [n, h+2, w+2, in_ld]; the conv reads channels [in_coff, in_coff+c_in) */
  int32_t in_ld, in_coff;
  const void* weight;    /* bf16 [c_out_pad, ksize*ksize*c_in], k index = (kh*ksize+kw)*c_in + c, BN folded */
  const float* bias;     /* fp32 [c_out_pad] */
  void* out;             /* padded NHWC bf16 [n, ho*u+2, wo*u+2, out_ld], u = 1+upsample; written at [out_coff, +c_out) */
  int32_t out_ld, out_coff;
  const void* res;       /* optional residual (NULL = none): padded NHWC bf16 with the conv-output geometry */
  int32_t res_ld, res_coff;
  int32_t upsample;      /* 1: replicate every output pixel 2x2 into `out` */
  float* out_f32;        /* Detect heads (NULL = off): fp32 pixel-major [n*ho*wo, out_f32_ld] instead of `out`;
                            columns [0, c_out_pad) of every row are written (pad columns = 0) */
  int32_t out_f32_ld;    /* >= c_out_pad, multiple of 4 */
  int32_t* err;          /* optional device int32 error word written by the in-kernel watchdog */
  int32_t weight_layout; /* Y3_W_*: how `weight` is packed (0 = tap-major as documented above) */
} y3_conv_desc;
int y3_conv_bn_act_fwd(const y3_conv_desc* d, y3_stream_t stream);
/* Input gradient of a STRIDE-2 3x3 conv (training; autograd of Conv.forward, models/common.py:71-75) as four parity-class
 * convolutions of the un-stuffed output gradient: `in` = dy, padded NHWC [n, h+2, w+2, in_ld] on the conv's OUTPUT grid (h, w =
 * output size), `weight` = the dgrad pack [c_in_pad rows = dx channels, 9 * c_dy] (taps flipped, y3_pack_weights), `out` = dx, padded
 * [n, 2h+2, 2w+2, out_ld]; `res` (optional, dx geometry) is added — pass `out` itself to accumulate.  ksize = 3, stride = 1 and
 * act = Y3_ACT_NONE in the descriptor (it describes the transposed conv on dy's grid). */
int y3_conv_dgrad_s2(const y3_conv_desc* d, y3_stream_t stream);
/* Weight layouts.  Y3_W_XPAIR (stride-2 3x3 with c_in in {16,32}, in_ld == c_in, in_coff == 0): bf16
 * [c_out_pad, 3, 2, 2, c_in] with element (kh, sp, par, c) = W[kh][2*sp+par][c] and zeros for the phantom column
 * 2*sp+par == 3 — two horizontally adjacent taps form one 2*c_in-channel GEMM k-block, which turns the 64-byte rows of
 * the thin first stride-2 layer (models/yolov3.yaml:19) into full 128-byte TMA rows.  y3_conv_weight_layout returns the
 * layout the kernel prefers for a descriptor's geometry (weight/bias/out pointers are not inspected); packing the
 * weights that way and setting weight_layout is optional — Y3_W_TAPS always works. */
#define Y3_W_TAPS 0
#define Y3_W_XPAIR 1
int y3_conv_weight_layout(const y3_conv_desc* d);
/* The kernel variant y3_conv_bn_act_fwd would launch for a descriptor (host-only query: pointers are checked for
 * alignment but never dereferenced, no tensor map is encoded, no GPU needed): tile shape, CTA pairs (cta_group::2), TMA-store
 * epilogue, halo reuse (one A box per filter row), weights resident in shared memory, epilogue warp groups, x-paired
 * stride-2 weights, tile counts and grid.  For tests and for reading the selection heuristics off a model. */
typedef struct y3_conv_plan_info {
  int32_t block_n, block_k, pair, staged, halo, resident_weights, epilogue_groups, xpair;
  int32_t m_tiles, n_tiles, k_blocks, grid;
} y3_conv_plan_info;
int y3_conv_plan(const y3_conv_desc* d, y3_conv_plan_info* out);
/* Tile N the kernel will use for c_out (weights/bias must be padded to a multiple of it). */
int y3_conv_cout_pad(int32_t c_out);

/* First layer: 3x3 stride-1 pad-1 conv on the NCHW image (c_in = 3), folded BN + SiLU, writing padded NHWC bf16.
 * Replaces Conv.forward_fuse for layer 0 together with the caller-side `im.float() / 255` (detect.py:187-191,
 * val.py:358-359) and the NCHW->NHWC/bf16 conversion.  c_out in {16, 32}.
 * weight: fp32 [27, c_out] (k = (c*3+kh)*3+kw), bias fp32 [c_out]. */
#define Y3_IN_F32 0
#define Y3_IN_U8 1
typedef struct y3_first_desc {
  const void* in;        /* [n, 3, h, w] fp32 or uint8 */
  int32_t in_dtype;      /* Y3_IN_* */
  float in_div;          /* > 0: pixel = value / in_div (255 for uint8 images); 0: use as is */
  int32_t n, h, w;
  const float* weight;
  const float* bias;
  int32_t c_out;
  void* out;             /* padded NHWC bf16 [n, h+2, w+2, out_ld] */
  int32_t out_ld, out_coff;
} y3_first_desc;
int y3_conv_first_fwd(const y3_first_desc* d, y3_stream_t stream);

/* Max-pool on padded NHWC bf16 (nn.MaxPool2d of yolov3-tiny.yaml; SPP pools, models/common.py:279,290).
 * Window of output (y,x) = input rows [y*stride+off, +k) x cols [x*stride+off, +k); out-of-image elements are ignored
 * (-inf padding) unless oob_zero, where they count as 0 (ZeroPad2d followed by MaxPool2d). */
typedef struct y3_pool_desc {
  const void* in;
  int32_t in_ld, in_coff;
  void* out;
  int32_t out_ld, out_coff;
  int32_t n, h, w, c;    /* input size (unpadded), channels (multiple of 8) */
  int32_t ho, wo;
  int32_t k, stride, off, oob_zero;
} y3_pool_desc;
int y3_maxpool_fwd(const y3_pool_desc* d, y3_stream_t stream);
/* Training mode (SPP, models/common.py:281-290, under autograd): the forward also records idx[n, ho, wo, c] (uint8) =
 * dy*k + dx of the first maximum in row-major window order — the element torch.nn.MaxPool2d back-propagates to — and the
 * backward gathers dIn[p] (+)= sum of dOut over the windows whose argmax is p (no atomics).  For y3_maxpool_bwd the
 * descriptor's `in` is dOut (geometry ho x wo), `out` is dIn (geometry h x w); oob_zero windows are not supported. */
int y3_maxpool_train_fwd(const y3_pool_desc* d, uint8_t* idx, y3_stream_t stream);
int y3_maxpool_bwd(const y3_pool_desc* d, const uint8_t* idx, int32_t accumulate, y3_stream_t stream);

/* Layout helpers (tests / feeding intermediate tensors): NCHW fp32 <-> padded NHWC bf16 channel slice. */
int y3_nchw_to_padded_nhwc(const float* src, int32_t n, int32_t c, int32_t h, int32_t w, void* dst, int32_t dst_ld,
                           int32_t dst_coff, y3_stream_t stream);
int y3_padded_nhwc_to_nchw(const void* src, int32_t src_ld, int32_t src_coff, int32_t n, int32_t c, int32_t h,
                           int32_t w, float* dst, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Detect decode.  Replaces the eval branch of Detect.forward and _make_grid (models/yolo.py:100-123):
 * z[b, off_l + (a*ny + y)*nx + x, :] = (xy: (2*sig + grid - 0.5)*stride, wh: (2*sig)^2 * anchor_px, rest: sig).
 */
#define Y3_MAX_LEVELS 5
#define Y3_MAX_ANCHORS 6
typedef struct y3_detect_level {
  const float* raw;                 /* y3_detect_decode_fwd: fp32 [bs, na, ny, nx, no] logits (the reference's x[i]) */
  const float* head;                /* y3_detect_head_decode_fwd: head-conv output, fp32 [bs*ny*nx, head_ld],
                                       column a*no + k (y3_conv_desc.out_f32) */
  int32_t head_ld;
  float* raw_out;                   /* y3_detect_head_decode_fwd: optional fp32 [bs, na, ny, nx, no] (models/yolo.py:98) */
  int32_t ny, nx;
  float stride;                     /* Detect.stride[i] */
  float anchor_w[Y3_MAX_ANCHORS];   /* anchors[i] * stride[i], pixels (anchor_grid, models/yolo.py:122) */
  float anchor_h[Y3_MAX_ANCHORS];
} y3_detect_level;
int y3_detect_decode_fwd(const y3_detect_level* levels, int32_t nl, int32_t bs, int32_t na, int32_t no, float* z,
                         y3_stream_t stream);
typedef struct y3_decode_desc {
  y3_detect_level levels[Y3_MAX_LEVELS];
  int32_t nl, bs, na, no;
  float* z;                         /* [bs, sum_l na*ny*nx, no] or NULL (training: logits only) */
} y3_decode_desc;
/* Fused head transpose + decode used by the graph executor: one pass from the head convs' pixel-major fp32 output to
 * z and to the reference-layout logits. */
int y3_detect_head_decode_fwd(const y3_decode_desc* d, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched NMS.  Replaces non_max_suppression (utils/general.py:630-750) incl. torchvision.ops.nms (:733) for nm=0;
 * autolabel priors (labels=, :689-695) are appended to `pred` by the caller as obj = 1 / one-hot rows.  Sync-free: results are padded device arrays plus per-image counts.
 *   pred      fp32 [bs, n_rows, 5+nc]  (xywh, obj, cls...)
 *   out       fp32 [bs, max_det, 6]    rows (x1,y1,x2,y2,conf,cls) sorted by conf desc, zero beyond out_count[b]
 *   out_src   int32 [bs, max_det, 2]   optional (pred row, class) of every kept detection
 *   out_count int32 [bs]
 *   overflow  int32 [bs]               optional; non-zero = candidates found (> cap): rerun with a larger capacity
 * The wall-clock time_limit break of the reference (:675,746-748) is intentionally not reproduced.
 */
typedef struct y3_nms_params {
  int32_t bs, n_rows, nc;
  float conf_thres, iou_thres;      /* must lie in [0,1] (the reference asserts, :658-659) */
  int32_t multi_label, agnostic;
  int32_t max_det;                  /* :734 */
  int32_t max_nms;                  /* 30000 (:674); <= 32768 */
  float max_wh;                     /* 7680 (:673) */
  int32_t cap;                      /* per-image candidate capacity, power of two >= 4096 */
  const int32_t* classes;           /* HOST array of class ids to keep (:717-718), or NULL */
  int32_t n_classes;
} y3_nms_params;
int32_t y3_nms_default_capacity(int32_t n_rows, int32_t nc, int32_t multi_label);
int64_t y3_nms_workspace_bytes(int32_t bs, int32_t cap);
int y3_nms_batched(const float* pred, const y3_nms_params* params, void* workspace, int64_t workspace_bytes, float* out,
                   int32_t* out_src, int32_t* out_count, int32_t* overflow, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Pairwise IoU.  Replaces box_iou (ultralytics; re-exported utils/metrics.py:10, used val.py:176): xyxy boxes,
 * out[i*m + j] = inter / (area1 + area2 - inter + eps).  box1 [n,4], box2 [m,4] fp32, 16-byte aligned. */
int y3_box_iou(const float* box1, int32_t n, const float* box2, int32_t m, float eps, float* out, y3_stream_t stream);
/* scale_boxes + clip_boxes (utils/general.py:613-626; callers detect.py:218, val.py:381-385): in place on columns 0..3
 * (xyxy) of n rows of `row_stride` floats: v = clamp((v - pad) / gain, 0, max) with pad_x/max_x for x1,x2 and pad_y/max_y
 * for y1,y2; gain = 1, pad = 0 gives clip_boxes. */
int y3_scale_boxes(float* boxes, int64_t n, int32_t row_stride, float pad_x, float pad_y, float gain, float max_x,
                   float max_y, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Training loss, forward + backward.  Replaces ComputeLoss.__call__ / build_targets (utils/loss.py:131-244) with
 * bbox_iou(CIoU) and BCEWithLogitsLoss(pos_weight), for fl_gamma = 0, autobalance off, gr = 1 (the shipped hyps).
 *   p[l]     fp32 [bs, na, ny_l, nx_l, nc+5] raw logits (train-mode Detect output, models/yolo.py:110)
 *   grad[l]  same shape (or NULL): receives d(out[0])/dp[l] * grad_scale
 *   targets  fp32 [nt, 6] = (image, class, x, y, w, h) normalised (collate_fn, utils/dataloaders.py:825-830)
 *   out      fp32 [4] = ((lbox+lobj+lcls)*bs, lbox, lobj, lcls)   (loss.py:181)
 */
typedef struct y3_loss_desc {
  int32_t nl, bs, na, nc;
  const float* p[Y3_MAX_LEVELS];
  float* grad[Y3_MAX_LEVELS];
  int32_t ny[Y3_MAX_LEVELS], nx[Y3_MAX_LEVELS];
  float anchors[Y3_MAX_LEVELS][Y3_MAX_ANCHORS][2]; /* Detect.anchors, grid units */
  const float* targets;
  int32_t nt;
  float box, obj, cls;       /* hyp gains (already rescaled as train.py:326-329) */
  float cls_pw, obj_pw;      /* BCE pos_weight */
  float anchor_t;
  float cp, cn;              /* smooth_bce(label_smoothing) targets */
  float balance[Y3_MAX_LEVELS];
  float grad_scale;          /* upstream gradient of out[0] (1 for loss.backward()) */
} y3_loss_desc;
int64_t y3_loss_workspace_bytes(const y3_loss_desc* d);
int y3_loss_fwd_bwd(const y3_loss_desc* d, void* workspace, int64_t workspace_bytes, float* out, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Training-mode Conv block (models/common.py:71-75 with BatchNorm2d in train mode) and its backward.  The convolution
 * (forward; dgrad = convolution with the transposed, tap-flipped weights) is y3_conv_bn_act_fwd with zero bias and
 * Y3_ACT_NONE; these entry points are the bandwidth-bound parts around it.  All activations: padded NHWC bf16 slices.
 */
/* Two-stage, atomic-free (bit-reproducible) reductions: a first-stage kernel writes one partial row per block into a
 * caller-owned workspace [y3_bn_partial_blocks(n, h, w, c)][width], a fixed-order second stage adds the rows. */
int32_t y3_bn_partial_blocks(int32_t n, int32_t h, int32_t w, int32_t c);  /* c = 0: one unit per image row (head gradient) */
/* per-channel sum and sum of squares of the conv output y over its n*h*w interior pixels:
 * partial[blocks][2][c] = (sum | sumsq).  c: power of two in [8, 2048]. */
int y3_bn_stats(const void* y, int32_t ld, int32_t coff, int32_t c, int32_t n, int32_t h, int32_t w, float* partial,
                y3_stream_t stream);
/* out[j] (+)= sum_b partial[b][j] for j < width, rows added in index order (SyncBatchNorm: sums before the all-reduce) */
int y3_colreduce_f32(const float* partial, int32_t nblk, int32_t width, float* out, int32_t accumulate, y3_stream_t stream);
/* batch statistics (given as nblk partial rows [2][c]; nblk = 1: already reduced) -> scale = gamma*rstd, shift = beta -
 * mean*scale, saved mean/rstd; running stats updated in place with the unbiased variance when non-NULL (nn.BatchNorm2d
 * semantics).  count = pixels behind the sums (n*h*w, times the world size under SyncBatchNorm). */
int y3_bn_finalize(const float* partial, int32_t nblk, const float* gamma, const float* beta, int32_t c, float count,
                   float eps, float momentum, float* scale, float* shift, float* mean, float* rstd, float* running_mean,
                   float* running_var, y3_stream_t stream);
typedef struct y3_bn_act_desc {
  const void* y;   int32_t y_ld, y_coff;       /* conv output (pre-BN) */
  const void* res; int32_t res_ld, res_coff;   /* optional residual added after the activation (Bottleneck shortcut) */
  void* out;       int32_t out_ld, out_coff;   /* a = SiLU(y*scale+shift) (+res); [n, h*u+2, w*u+2, out_ld], u = 1+upsample */
  const float* scale; const float* shift;
  int32_t n, h, w, c, upsample;
} y3_bn_act_desc;
int y3_bn_act_fwd(const y3_bn_act_desc* d, y3_stream_t stream);
typedef struct y3_bn_bwd_desc {
  const void* y;  int32_t y_ld, y_coff;        /* saved conv output */
  const void* da; int32_t da_ld, da_coff;      /* gradient w.r.t. the block output (2x geometry when upsample) */
  void* dy;       int32_t dy_ld, dy_coff;      /* gradient w.r.t. the conv output (input of dgrad / wgrad) */
  const float* scale; const float* shift; const float* mean; const float* rstd;
  float* sums;       /* [2][c] = (sum dz | sum dz*xhat): phase 0/1 out, phase 2 in (the all-reduced sums) */
  float* partial;    /* workspace [y3_bn_partial_blocks(n, h, w, c)][2][c] of the reduction phase (phases 0, 1) */
  float* dbeta_acc;  /* optional [c]: += sum dz      (the bn.bias gradient, accumulated like autograd does) */
  float* dgamma_acc; /* optional [c]: += sum dz*xhat (the bn.weight gradient) */
  int32_t n, h, w, c, upsample;
  int32_t phase;   /* 0: sums then apply (single GPU); 1: sums only; 2: apply only — SyncBatchNorm (train.py:270-272) puts
                      an all-reduce of the two sums between 1 and 2 */
  float count;     /* pixels behind the sums used by the apply phase (all ranks); 0 = this rank's n*h*w */
} y3_bn_bwd_desc;
int y3_bn_act_bwd(const y3_bn_bwd_desc* d, y3_stream_t stream);
/* fp32 master weights [co, ci, k, k] -> bf16 forward pack [co_pad, k*k*ci] and/or dgrad pack [ci_pad, k*k*co] (taps
 * flipped, channels swapped); pad rows must already be zero */
int y3_pack_weights(const float* w, int32_t co, int32_t ci, int32_t k, void* fwd, void* dgrad, y3_stream_t stream);
/* Batched form used by the training engine: the fp32 masters live in ONE flat buffer with every conv weight stored
 * [co][kh][kw][ci] (channels_last strides of the [co,ci,k,k] parameter == the forward pack's order), so
 *   y3_f32_to_bf16        converts the whole buffer once per step (forward packs are views of the copy), and
 *   y3_pack_dgrad_batched transposes every layer of a device-resident table into its dgrad pack in one launch. */
int y3_f32_to_bf16(const float* src, void* dst, int64_t n, y3_stream_t stream);
typedef struct y3_pack_item {
  int64_t src_off;   /* element offset of this layer's [co_rows][k*k][ci] weights inside the bf16 flat copy */
  void* dst;         /* dgrad pack, bf16 [ci_pad][k*k][dst_co] (rows >= ci stay zero) */
  int32_t co_rows;   /* rows present in the source (c_out, or the padded 256 of a Detect head) */
  int32_t ci, k;
  int32_t dst_co;    /* row pitch of the pack = c_out the dgrad conv reduces over */
  int32_t tile_begin;/* first 32x32 transpose tile of this layer: k*k * ceil(co_rows/32) * ceil(ci/32) tiles each, consecutive */
  int32_t reserved;
} y3_pack_item;
int y3_pack_dgrad_batched(const y3_pack_item* items_dev, int32_t n_items, const void* wbf, int32_t total_tiles,
                          y3_stream_t stream);
/* Detect-head gradient: g = dL/draw fp32 [n, na, ny, nx, no] (ComputeLoss output) -> dy bf16 padded NHWC channel a*no+o
 * (the head conv's output order; channels >= na*no zeroed) and partial[y3_bn_partial_blocks(n, ny, 0, 0)][256] column sums
 * (bias gradient = y3_colreduce_f32 over them). */
int y3_head_grad_pack(const float* g, int32_t n, int32_t na, int32_t ny, int32_t nx, int32_t no, void* dy, int32_t dy_ld,
                      int32_t dy_coff, float* partial, y3_stream_t stream);
/* dy of a stride-2 conv scattered onto the even positions of a zeroed [n, 2ho+2, 2wo+2, dst_ld] buffer */
int y3_zero_stuff(const void* src, int32_t src_ld, int32_t src_coff, void* dst, int32_t dst_ld, int32_t dst_coff, int32_t n,
                  int32_t ho, int32_t wo, int32_t c, y3_stream_t stream);
/* dW[co, ci, kh, kw] += sum_p dy[p, co] * x[p + shift(kh,kw), ci] on the stride-1 padded grid [n, h+2, w+2]; dw is fp32,
 * zeroed by the caller; co, ci multiples of 8.  dw_layout Y3_DW_OIHW: PyTorch's [co, ci, k, k].  Y3_DW_TAP_MAJOR:
 * [k*k, co, ci] — every (tap, co) row is contiguous in ci, so the tensor-core kernel accumulates with 16-byte vector
 * reductions instead of one 4-byte atomic per element (the scattered atomics, ~45 G/s, were all of its time); the caller
 * permutes once when it hands the gradient to the optimizer.  Needs c_in % 32 == 0 (y3_conv_wgrad_tap_major tells). */
#define Y3_DW_OIHW 0
#define Y3_DW_TAP_MAJOR 1
#define Y3_DW_OHWI 2       /* [co, k*k, ci] == the channels_last strides of a [co, ci, k, k] tensor: the training engine's
                              flat gradient buffer (the gradient IS the parameter's .grad view, no permute) */
typedef struct y3_wgrad_desc {
  const void* dy; int32_t dy_ld, dy_coff;
  const void* x;  int32_t x_ld, x_coff;
  float* dw;
  int32_t co, ci, ksize, n, h, w;
  int32_t dw_layout;
  int32_t accumulate;     /* 1: dw holds earlier contributions that must be kept (always reduce, never plain-store) */
  int32_t deterministic;  /* 1: no split over pixels — one CTA per dW tile, bit-reproducible, slower on the early layers */
  int32_t stride;         /* 0/1: dy on x's grid (a stride-2 conv passes the zero-stuffed dy).  2: DIRECT stride-2 — dy is the
                             conv's own [n, h/2+2, w/2+2, dy_ld] output-grid gradient, x is read through its row/column parity view;
                             3x3 only, needs y3_conv_wgrad_s2_supported(h, w) and c_in % 32 == 0 */
} y3_wgrad_desc;
int y3_conv_wgrad(const y3_wgrad_desc* d, y3_stream_t stream);
/* 1 if the direct stride-2 form (stride = 2) can tile an input of h x w (an 80-pixel tw x th patch must divide the output) */
int y3_conv_wgrad_s2_supported(int32_t h, int32_t w);
/* 1 if y3_conv_wgrad accepts Y3_DW_TAP_MAJOR for this c_in (the tcgen05 kernel is in use), else 0 */
int y3_conv_wgrad_tap_major(int32_t c_in);
/* dst (+)= src over the interior pixels of two padded NHWC bf16 slices of equal [n,h,w,c] (gradient fan-in) */
int y3_add_nhwc(const void* src, int32_t src_ld, int32_t src_coff, void* dst, int32_t dst_ld, int32_t dst_coff, int32_t n,
                int32_t h, int32_t w, int32_t c, int32_t accumulate, y3_stream_t stream);
/* 3x3 pad-1 im2col of the [n,3,h,w] image (Y3_IN_F32 | Y3_IN_U8, optional /in_div) into 32 bf16 channels of a padded
 * NHWC buffer, column (c*3+kh)*3+kw; lets training run layer 0 as a 1x1 conv with the generic kernels */
int y3_im2col_first(const void* in, int32_t in_dtype, float in_div, int32_t n, int32_t h, int32_t w, void* out,
                    int32_t out_ld, int32_t out_coff, y3_stream_t stream);
/* out[c] += sum over rows of g[row, c] (fp32 pixel-major; Detect-head bias gradients) */
int y3_colsum_f32(const float* g, int32_t ld, int32_t c, int64_t rows, float* out, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Image pre-processing on the device (SURVEY §8(f) row f1): letterbox (utils/augmentations.py:104-134: cv2.resize
 * INTER_LINEAR to new_w x new_h, then a constant border) fused with the HWC->CHW / BGR->RGB step of the loaders
 * (utils/dataloaders.py:308-310).  src: uint8 [src_h, src_w, 3] with row pitch src_pitch bytes (a decoded BGR frame);
 * dst: uint8 [out_h, out_w, 3] (out_chw = 0) or [3, out_h, out_w] (out_chw = 1), channel order reversed when swap_rb.
 * The resized image sits at (top, left); everything else is pad[] (given in SOURCE channel order, 114 in the reference).
 * The resize reproduces OpenCV's 8-bit INTER_LINEAR bit for bit (incl. its 2x-shrink INTER_AREA shortcut and the plain copy
 * when no resize is needed).  The geometry (new size, offsets) is the caller's: letterbox's scalar arithmetic stays on the host. */
typedef struct y3_letterbox_desc {
  const void* src; int32_t src_h, src_w, src_pitch;
  int32_t new_h, new_w, top, left;
  void* dst;       int32_t out_h, out_w;
  int32_t out_chw, swap_rb;
  uint8_t pad[4];
} y3_letterbox_desc;
int y3_letterbox_u8(const y3_letterbox_desc* d, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Test-time augmentation (Model._forward_augment, models/yolo.py:239-280).
 * y3_scale_img_f32: scale_img (ultralytics; yolo.py:246) — bilinear (align_corners = false) resample of fp32 [n,c,h,w] (read
 *   left-right flipped when flip_lr) to rh x rw inside an [n,c,oh,ow] output whose right / bottom remainder is pad_value (0.447).
 * y3_tta_merge: rows [row_begin, row_end) of one view's decoded z [bs, rows, no] go to rows [out_row_off, ...) of the merged
 *   output [bs, out_rows, no] with _descale_pred applied (xywh /= scale; x = img_w - x when the view was flipped): the
 *   _clip_augmented row selection and the torch.cat of the reference are the addressing of this copy. */
int y3_scale_img_f32(const float* in, int32_t n, int32_t c, int32_t h, int32_t w, int32_t rh, int32_t rw, int32_t oh, int32_t ow,
                     int32_t flip_lr, float pad_value, float* out, y3_stream_t stream);
int y3_tta_merge(const float* z, int32_t bs, int32_t rows, int32_t no, int32_t row_begin, int32_t row_end, float scale,
                 int32_t flip_lr, float img_w, float* out, int32_t out_rows, int32_t out_row_off, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Validation matching (val.process_batch, val.py:147-188) for a whole batch and all IoU thresholds in one launch.
 * det: [bs, det_stride, 6] rows (x1,y1,x2,y2,conf,cls) in confidence order (the NMS output), det_count[bs] valid rows per image
 * (NULL: max_det each); labels: [nl, 6] rows (image, cls, x1,y1,x2,y2) in the same coordinate space as det; iouv: [niou]
 * thresholds (val.py:301: linspace(0.5, 0.95, 10)).  correct[bs, max_det, niou] (bytes 0/1):
 *   correct[d, t] = 1  <=>  detection d's best same-class label l (IoU >= iouv[t], highest IoU) exists and d is the
 *   lowest-index detection whose best label is l  — the result of the reference's sort / np.unique / np.unique sequence.
 * IoU = inter / (area_label + area_det - inter + eps), the reference box_iou's fp32 operation order (eps 1e-7).
 * At most 1024 labels per image are matched; overflow[bs] (optional) reports how many were ignored. */
int y3_val_match(const float* det, const int32_t* det_count, int32_t bs, int32_t max_det, int32_t det_stride,
                 const float* labels, int32_t nl, const float* iouv, int32_t niou, float eps, uint8_t* correct,
                 int32_t* overflow, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Validation metrics (csrc/y3_metrics.cu).
 * y3_ap_per_class: ap_per_class + compute_ap (utils/metrics.py:22-120, val.py:424-426).  Row i (0 <= i < n) is
 *   (conf[i * conf_stride], cls[i * cls_stride], tp[i * niou + 0..niou)); with det_count, row i is valid iff
 *   i % rows_per_image < det_count[i / rows_per_image] (the padded nms_batched / process_batch_batched layout read in place),
 *   without it every row is.  Target classes: target_cls[k * target_stride], k < n_targets.  Classes are integral values in
 *   [0, nc); others are counted in status and ignored.  Outputs are indexed by class id: ap[nc, niou], p, r, f1, tp_out, fp_out
 *   [nc] (float64, at the F1 index), nt[nc] label counts, present[nc] (the class occurs in the targets: the reference's
 *   unique_classes; other rows are zero), f1_index[1], status[3] = (valid rows with a bad class, targets with a bad class,
 *   curves whose true positives exceed their labels: outside the reference's contract, their AP is unspecified).
 *   Order: class, conf descending, then row — stable, where the reference's argsort is not (bit-equal confidences).
 *   AP is bit-identical to the reference (np.interp and numpy's pairwise trapezoid restated in double, no contraction);
 *   p / r / f1 differ at most by the reference's smooth(), which sums through BLAS.  niou <= 64, nc <= 65535.
 *   workspace: >= y3_ap_per_class_workspace_bytes(n, n_targets, niou, nc) bytes (device). */
int64_t y3_ap_per_class_workspace_bytes(int64_t n, int64_t n_targets, int32_t niou, int32_t nc);
int y3_ap_per_class(const float* conf, int64_t conf_stride, const float* cls, int64_t cls_stride, const uint8_t* tp, int32_t niou,
                    int64_t n, const int32_t* det_count, int64_t rows_per_image, const float* target_cls, int64_t target_stride,
                    int64_t n_targets, int32_t nc, double eps, void* workspace, int64_t workspace_bytes, double* ap, double* p,
                    double* r, double* f1, double* tp_out, double* fp_out, int64_t* nt, uint8_t* present, int32_t* f1_index,
                    int32_t* status, y3_stream_t stream);
/* y3_confusion_update: ConfusionMatrix.process_batch (utils/metrics.py:134-178) for every image of a padded batch, accumulated
 *   into matrix[(nc+1) * (nc+1)] (int64, [pred][true], background last; integer atomics).  det [bs, det_stride, 6] (xyxy, conf,
 *   cls) + det_count[bs] (NULL: max_det each; <= 0: the detections=None call), labels [nl, 6] = (image, cls, xyxy).  Detections
 *   with conf > conf_thres; pairs with IoU > iou_thres (y3_val_match's IoU, eps 1e-7); each detection keeps its best label, each
 *   label its best detection among those (bit-equal IoU: lower label, then lower detection index).  Unmatched detections count
 *   as background only when the image has a match (the reference's quirk).  Class ids are truncated (tensor.int()); ids outside
 *   [0, nc) are counted in status[0], labels beyond 1024 in one image in status[1] (both accumulate). */
int y3_confusion_update(const float* det, const int32_t* det_count, int32_t bs, int32_t max_det, int32_t det_stride,
                        const float* labels, int32_t nl, int32_t nc, float conf_thres, float iou_thres, float eps, int64_t* matrix,
                        int32_t* status, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Optimizer step over ONE flat fp32 parameter buffer (train.py:411-421: clip_grad_norm_(10.0), SGD-nesterov with the three
 * parameter groups of smart_optimizer utils/torch_utils.py:207-237, ModelEMA.update) — csrc/y3_optim.cu.
 * Layout contract: every parameter occupies a slot whose length is a multiple of 256 elements; group[i] is the group of
 * elements [256 i, 256 i + 256): 0 = weights with decay, 1 = BatchNorm weights, 2 = biases, >= 3 = not trained (buffers).
 * hp_dev: DEVICE float[11] = lr[3], weight_decay[3], momentum, nesterov, max_norm (0: no clipping), ema decay of this
 * update, gradient pre-scale (1/world_size after a SUM all-reduce) — read at run time, so the launches can sit in a CUDA
 * graph while the scheduler changes them.
 */
int32_t y3_sumsq_blocks(void);  /* floats of workspace y3_grad_sumsq needs */
/* out[0] = sum g[i]^2 (two-stage, fixed order: bit-reproducible); n % 4 == 0 */
int y3_grad_sumsq(const float* g, int64_t n, float* partial, float* out, y3_stream_t stream);
/* p, m (momentum buffer, zero-initialised), ema (optional) updated in place from g; gsumsq (from y3_grad_sumsq) is read
 * only when hp_dev[8] > 0.  n = elements of p (and of ema); g and m are only touched where group < 3. */
int y3_sgd_step(float* p, const float* g, float* m, float* ema, const uint8_t* group, int64_t n, const float* hp_dev,
                const float* gsumsq, y3_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Whole-graph executor.  Replaces BaseModel._forward_once (models/yolo.py:135-147): the Python loop over nn.Modules
 * becomes an immutable list of prepared launches (TMA descriptors encoded once at create) replayed on one stream.
 * All buffers belong to the caller; y3_model_forward is CUDA-graph capturable.
 */
#define Y3_OP_CONV_FIRST 1
#define Y3_OP_CONV 2
#define Y3_OP_MAXPOOL 3
#define Y3_OP_DECODE 4
typedef struct y3_op {
  int32_t kind;          /* Y3_OP_*: selects which member below is read */
  y3_conv_desc conv;
  y3_first_desc first;
  y3_pool_desc pool;
  y3_decode_desc decode;
} y3_op;
typedef struct y3_model y3_model;
int y3_model_create(const y3_op* ops, int32_t n_ops, y3_model** out);
/* input: optional override of the first op's image pointer (NULL = the pointer given at create). */
int y3_model_forward(const y3_model* m, const void* input, y3_stream_t stream);
int32_t y3_model_num_launches(const y3_model* m);
/* Profiling aid (synchronises; not capturable): average device time of every launch over `iters` passes, measured
 * with CUDA events on `stream`; ms_out is a HOST array of y3_model_num_launches() floats. */
int y3_model_forward_timed(const y3_model* m, const void* input, y3_stream_t stream, float* ms_out, int32_t iters);
void y3_model_destroy(y3_model* m);

#ifdef __cplusplus
}
#endif
#endif /* YOLOV3_B200_H */
